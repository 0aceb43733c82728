"""GPU tests of scene updates (rh_scene_update / rh_multi_scene_update / Scene.update): after every edit of a chain on
every shipped scene the updated scene renders, answers queries and holds the light tables of a fresh rh_scene_create of
the edited description; only the tables an edit touches are rebuilt; the learned state follows the update's class;
accumulators refuse a state fixed before an update; failed updates leave the scene as it was; the multi-GPU replica
follows."""
import ctypes as C

import numpy as np
import pytest

import rayhs_b200 as rh
from rayhs_b200 import capi
from tests.test_trace_rays_gpu import has_transparent
from tests.util import SCENES, assert_parity, load_scene, oracle_for

pytestmark = pytest.mark.gpu

W, H, SPP, SEED = 96, 72, 4, 0x5CE7E
RAY_KEYS = ("rays_primary", "rays_reflect", "rays_probe", "rays_exit", "rays_shadow")
UPDATED_MSG = "the scene was updated since the"


class Fresh:
    """rh_scene_create of a Scene's current flat description: what an updated scene must be indistinguishable from."""

    def __init__(self, sc):
        self.flat_ptr = sc.flat
        self._flat_keep = sc
        self.device = C.c_void_p()
        rh.init()
        capi.check(capi.lib().rh_scene_create(self.flat_ptr, C.byref(self.device)))

    @property
    def flat(self):
        return self.flat_ptr

    def close(self):
        capi.lib().rh_scene_destroy(self.device)


def frame(scene, camera, max_depth, w=W, h=H, **kw):
    return rh.render(rh.Rendering(scene, camera, w, h, max_depth), spp=SPP, seed=SEED, want_hit_ids=True, **kw)


def tables(scene):
    t = rh.Scene.light_tables(scene)
    ms, info = (C.c_double * 3)(), (C.c_int32 * 4)()
    capi.check(capi.lib().rh_scene_info(scene.device, ms, info))
    b = (C.c_uint64 * 5)()
    capi.check(capi.lib().rh_scene_record_bytes(scene.device, b))
    return t, list(info), list(b)


def assert_same_tables(a, b, what):
    (ta, ia, ba), (tb, ib, bb) = a, b
    assert ia == ib and ba == bb, (what, ia, ib, ba, bb)
    assert ta["res"] == tb["res"] and np.array_equal(ta["index"], tb["index"]), what
    assert ta["maps"].shape == tb["maps"].shape and ta["maps"].tobytes() == tb["maps"].tobytes(), what
    assert (ta["lit"] is None) == (tb["lit"] is None), what
    if ta["lit"] is not None:
        assert np.array_equal(ta["lit"], tb["lit"]), what


def assert_same_frame(got, want, forks, what):
    assert np.array_equal(got.hit_ids, want.hit_ids), what
    assert {k: got.stats[k] for k in RAY_KEYS} == {k: want.stats[k] for k in RAY_KEYS}, what
    if forks:
        assert_parity(got.pixels, want.pixels, what)
    else:
        assert np.array_equal(got.pixels, want.pixels), what


def mesh_material(sc):
    raw = sc.raw.contents
    for i in range(raw.n_objects):
        if raw.objects[i].kind == capi.RH_OBJ_MESH:
            return raw.objects[i].material
    return None


def edit_chain(sc):
    """(label, materials, lights) edits applied one after the other, each from the tables the previous one left."""
    cam = np.array(sc.camera.position[:])

    def colours(m, l):
        for x in m:
            x.color1[:] = [0.8 * c for c in x.color1]
            x.color2[:] = [0.5 + 0.5 * c for c in x.color2]
        for x in l:
            x.color[:] = [0.7 * c for c in x.color]
            x.radius *= 1.5
        return m, l

    def move_point(m, l):
        pts = [i for i in range(len(l)) if l[i].kind == capi.RH_LIGHT_POINT] or list(range(len(l)))
        if pts:
            l[pts[0]].vec[:] = [v + d for v, d in zip(l[pts[0]].vec, (0.37, 0.21, -0.29))]
        return m, l

    def point_to_directional(m, l):
        pts = [i for i in range(len(l)) if l[i].kind == capi.RH_LIGHT_POINT]
        if pts:
            l[pts[-1]].kind = capi.RH_LIGHT_DIRECTIONAL
            l[pts[-1]].vec[:] = (0.3, -1.0, 0.45)
        return m, l

    def add_light(m, l):
        x = capi.rh_light()
        x.kind = capi.RH_LIGHT_POINT
        x.vec[:] = cam + np.array([0.4, 1.3, 0.2])
        x.color[:] = (0.3, 0.3, 0.25)
        x.radius = 1.0
        return m, list(l) + [x]

    def remove_light(m, l):
        return m, list(l)[1:]

    def first_kind(kind, to, ior=None):
        def f(m, l):
            for x in m:
                if x.kind == kind:
                    x.kind = to
                    if to == capi.RH_MAT_TRANSPARENT:
                        x.ior = 1.45 if ior is None else ior
                    break
            return m, l
        return f

    mm = mesh_material(sc)

    def emmit(on, saved={}):
        def f(m, l):
            if mm is None:
                return m, l
            if on:
                saved["m"] = capi.rh_material.from_buffer_copy(m[mm])
                m[mm].kind = capi.RH_MAT_EMMIT
                m[mm].color1[:] = (0.9, 0.6, 0.3)
            else:
                m[mm] = saved["m"]
            return m, l
        return f

    return [("colours", colours), ("move_point", move_point), ("point_to_directional", point_to_directional),
            ("add_light", add_light), ("remove_light", remove_light),
            ("diffuse_to_mirror", first_kind(capi.RH_MAT_DIFFUSE, capi.RH_MAT_MIRROR)),
            ("plastic_to_transparent", first_kind(capi.RH_MAT_PLASTIC, capi.RH_MAT_TRANSPARENT)),
            ("mesh_to_emmit", emmit(True)), ("mesh_back", emmit(False))]


@pytest.mark.parametrize("name", SCENES)
def test_every_edit_equals_a_fresh_scene(name):
    sc = load_scene(name)
    sc.device
    oracle_done = False
    for label, edit in edit_chain(sc):
        m, l = edit(sc.materials, list(sc.lights))
        info = sc.update(materials=m, lights=l)
        fresh = Fresh(sc)
        try:
            what = f"{name}/{label}"
            forks = has_transparent(sc)
            assert_same_tables(tables(sc), tables(fresh), what)
            assert_same_frame(frame(sc, sc.camera, sc.max_depth), frame(fresh, sc.camera, sc.max_depth), forks, what)
            if label == "colours":
                assert info["colours_only"] == 1 and info["maps_rasterised"] == 0 and info["lit_queries"] == 0, (what, info)
            # queries: closest hits, shadows towards every light (one index past the old table too), radiance
            rng = np.random.default_rng(3)
            n = 4096
            o = np.repeat(np.array(sc.camera.position[:])[None], n, 0)
            d = rng.normal(size=(n, 3))
            a, b = rh.closestIntersection(sc, o, d), rh.closestIntersection(fresh, o, d)
            assert a.records.tobytes() == b.records.tobytes(), what
            for li in range(len(sc.lights)):
                assert np.array_equal(rh.shadowIntersection(sc, li, o, d), rh.shadowIntersection(fresh, li, o, d)), what
            ra, rb = rh.traceRay(sc, o, d, 3), rh.traceRay(fresh, o, d, 3)
            if forks:
                assert np.allclose(ra.colors, rb.colors, rtol=1e-9, atol=1e-12), what
            else:
                assert np.array_equal(ra.colors, rb.colors), what
        finally:
            fresh.close()
        if not oracle_done and label in ("move_point", "diffuse_to_mirror"):
            # the updated scene against the oracle of Scene.raw, one sample at the pixel corner
            w, h = 48, 36
            gpu = rh.render(rh.renderingFromScene(sc, w, h), want_hit_ids=True)
            ref = oracle_for(sc).render(sc.camera, w, h, sc.max_depth)
            assert np.array_equal(gpu.hit_ids.reshape(-1, 2), ref["hit_ids"].reshape(-1, 2)), name
            assert_parity(gpu.pixels, ref["rgb_u8"], name)
            oracle_done = True


def test_incremental_rebuilds_on_dragon_low():
    sc = load_scene("dragon_low")
    lights = list(sc.lights)
    assert len(lights) == 3 and all(x.kind == capi.RH_LIGHT_POINT for x in lights)
    before = rh.Scene.light_tables(sc)
    n_meshes = int((before["index"] != 0xFFFFFFFF).any(axis=0).sum())
    kept_useful = int((before["index"][1:] != 0xFFFFFFFF).sum())
    n_slots = len(before["lit"]) if before["lit"] is not None else 0
    lights[0].vec[1] += 0.25
    info = sc.update(lights=lights)
    assert info["colours_only"] == 0 and info["occluders_rebuilt"] == 0
    # one raster per occluder mesh for the moved light (a mesh none of whose maps is useful is not in n_meshes)
    assert n_meshes <= info["maps_rasterised"] <= 8 and info["maps_kept"] == kept_useful, info
    assert 0 < info["lit_queries"] <= n_slots, info  # one light's queries on the meshes' slots
    m = sc.materials
    m[0].color1[:] = (0.1, 0.9, 0.1)
    info = sc.update(materials=m)
    assert info == {"colours_only": 1, "occluders_rebuilt": 0, "maps_rasterised": 0, "maps_kept": 0, "lit_queries": 0}
    mm = mesh_material(sc)
    m[mm].kind = capi.RH_MAT_EMMIT
    info = sc.update(materials=m)
    assert info["occluders_rebuilt"] == 1 and info["colours_only"] == 0


def test_learned_state_follows_the_update_class():
    sc = load_scene("dragon_low")
    small = rh.renderingFromScene(sc, 160, 90)
    job = rh.renderingFromScene(sc, 2400, 1350)
    frames = [rh.render(job) for _ in range(3)]
    assert [f.stats["shadow_split"] for f in frames] == [0, 0, 1]
    decided = rh.render(job).stats["shadow_split"]
    m = sc.materials
    m[0].color1[:] = (0.2, 0.4, 0.6)
    assert sc.update(materials=m)["colours_only"] == 1
    assert rh.render(small).stats["shadow_split"] == decided      # the decided schedule persists
    l = list(sc.lights)
    l[1].vec[0] -= 0.3
    sc.update(lights=l)
    assert rh.render(small).stats["shadow_split"] == 0             # undecided again: small frames pooled, not counted
    assert [rh.render(job).stats["shadow_split"] for _ in range(3)] == [0, 0, 1]


@pytest.mark.parametrize("kind", ["accum", "adaptive"])
def test_accumulators_refuse_a_state_fixed_before_an_update(kind):
    sc = load_scene("dragon_low")
    job = rh.renderingFromScene(sc, 64, 48)
    def make():
        if kind == "accum":
            acc = rh.Accumulator(job, stream_spp=16)
            return acc, lambda: acc.add(2, seed=SEED)
        acc = rh.AdaptiveAccumulator(job, stream_spp=16)
        return acc, lambda: acc.add(2, seed=SEED, threshold=0.0, min_spp=16)  # every pixel active in every call

    acc, add = make()
    add()
    assert sc.update() == {"colours_only": 0, "occluders_rebuilt": 0, "maps_rasterised": 0, "maps_kept": 0, "lit_queries": 0}
    add()                                          # a no-op update: accepted
    sc.update(materials=sc.materials)
    add()
    state = acc.state() if kind == "adaptive" else None
    m = sc.materials
    m[0].color1[:] = (0.9, 0.1, 0.1)
    sc.update(materials=m)
    with pytest.raises(capi.RayHsError, match=UPDATED_MSG):
        add()
    if kind == "adaptive":
        assert all(np.array_equal(x, y) for x, y in zip(state, acc.state()))
    else:
        assert acc.samples == 6
    acc.reset()
    got = [add() for _ in range(3)][-1]
    ref, ref_add = make()
    want = [ref_add() for _ in range(3)][-1]
    assert np.array_equal(got.pixels, want.pixels)
    ref.close()
    acc.close()


def test_failed_updates_leave_the_scene_as_it_was():
    sc = load_scene("cornellBox")
    sc.device
    before, tb = frame(sc, sc.camera, sc.max_depth), tables(sc)
    L = capi.lib()
    m, l = sc.materials, sc.lights
    n_m, n_l = len(m), len(l)

    def refused(mats, n_mats, lights, n_lights, text):
        assert L.rh_scene_update(sc.device, mats, n_mats, lights, n_lights, None) == capi.RH_ERR_ARG
        assert text in L.rh_last_error().decode()

    refused(m, n_m - 1, None, 0, "differs from the scene's material count")
    bad = (capi.rh_material * n_m).from_buffer_copy(m)
    bad[0].kind = 17
    refused(bad, n_m, None, 0, "unknown material kind")
    bad = (capi.rh_material * n_m).from_buffer_copy(m)
    bad[0].kind, bad[0].cmap_kind = capi.RH_MAT_DIFFUSE, 9
    refused(bad, n_m, None, 0, "unknown colour-map kind")
    bad[0].cmap_kind, bad[0].texture = capi.RH_CMAP_TEXTURE, 5
    refused(bad, n_m, None, 0, "texture index out of range")
    bad_l = (capi.rh_light * n_l).from_buffer_copy(l)
    bad_l[0].kind = 7
    refused(None, n_m, bad_l, n_l, "unknown light kind")
    assert L.rh_scene_update(None, m, n_m, l, n_l, None) == capi.RH_ERR_ARG
    after = frame(sc, sc.camera, sc.max_depth)
    assert np.array_equal(after.pixels, before.pixels) and np.array_equal(after.hit_ids, before.hit_ids)
    assert_same_tables(tables(sc), tb, "after refused updates")


def test_multi_scene_update_follows_the_single_scene():
    import torch

    n = torch.cuda.device_count()
    sc = load_scene("dragon_low")
    job = rh.renderingFromScene(sc, 160, 120)
    try:
        rh.render_multi(job, n, spp=2, seed=SEED)
        l = list(sc.lights)
        l[2].vec[2] += 0.4
        m = sc.materials
        m[0].kind = capi.RH_MAT_MIRROR
        sc.update(materials=m, lights=l)
        got = rh.render_multi(job, n, spp=2, seed=SEED)
        want = rh.render(job, spp=2, seed=SEED)
        assert np.array_equal(got.pixels, want.pixels)
    finally:
        rh.multi_shutdown([sc])
