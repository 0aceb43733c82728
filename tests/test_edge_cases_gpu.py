"""GPU parity on hand-built scenes that reach the code paths the shipped scenes do not: empty inputs,
Empty tree children, every material kind, both projections, > 32 lights (simple shadow kernel),
> 64 objects (tables read from global memory), deep recursion with Transparent forks, the synthetic C5 scene."""
import numpy as np
import pytest

import rayhs_b200 as rh
from oracle.orc import OracleScene
from tests.test_trace_rays_gpu import has_transparent
from tests.util import RawScene, assert_oracle_exact, grid_mesh, render_linear

pytestmark = pytest.mark.gpu


def both(rs, w, h, depth=None, spp=1, offsets=None, **kw):
    """Renders with either shadow schedule and holds both to the oracle: hit ids and ray counts equal, the image the
    oracle's by assert_oracle_exact.  Without a Transparent material the schedules give the same bytes and the same
    linear bits; with one, its forks add with atomics in any order (the 1-LSB wobble of DESIGN §3)."""
    depth = rs.max_depth if depth is None else depth
    job = rh.Rendering(rs, rs.camera, w, h, depth)
    img = render_linear(job, spp=spp, offsets=offsets, shadow="pooled", **kw)
    img_split = render_linear(job, spp=spp, offsets=offsets, shadow="split", **kw)
    assert np.array_equal(img.hit_ids, img_split.hit_ids), "hit ids must not depend on the shadow schedule"
    if has_transparent(rs):
        d = np.abs(img.pixels.astype(np.int32) - img_split.pixels.astype(np.int32))
        assert d.max() <= 1 and (d > 0).mean() < 1e-3, "pooled vs split schedule"
    else:
        assert np.array_equal(img.pixels, img_split.pixels), "pooled vs split schedule"
        assert np.array_equal(img.linear.view(np.uint64), img_split.linear.view(np.uint64)), "pooled vs split schedule"
    for k in ("rays_primary", "rays_reflect", "rays_probe", "rays_exit", "rays_shadow"):
        assert img.stats[k] == img_split.stats[k], k
    ref = OracleScene(rs.raw).render(rs.camera, w, h, depth, spp=spp, offsets=offsets)
    assert np.array_equal(img.hit_ids.reshape(h, w, spp, 2), ref["hit_ids"]), "hit ids"
    straddled = [assert_oracle_exact(i.pixels, i.linear, ref, what) for i, what in ((img, "pooled"), (img_split, "split"))]
    print("straddled channels", straddled)
    got = tuple(img.stats[k] for k in ("rays_primary", "rays_reflect", "rays_probe", "rays_exit", "rays_shadow"))
    want = tuple(ref["rays"][k] for k in ("primary", "reflect", "probe", "exit", "shadow"))
    assert got == want, (got, want)
    return img, ref


QUAD = dict(positions=[(-1, -1, 0), (1, -1, 0), (1, 1, 0), (-1, 1, 0)], normals=[(0, 0, -1)] * 4,
            uvs=[(0, 0), (1, 0), (1, 1), (0, 1)], indices=[0, 1, 2, 0, 2, 3])


def test_empty_scene_and_no_lights():
    rs = RawScene([], [{"kind": "diffuse"}], [])
    img, _ = both(rs, 33, 17)
    assert not img.pixels.any()
    rs = RawScene([{"kind": "sphere", "center": (0, 0, 0), "radius": 1.0}], [{"kind": "diffuse", "color1": (0.5, 1.0, 2.0)}], [])
    img, _ = both(rs, 40, 40)
    assert tuple(img.pixels[20, 20]) == (25, 51, 102)  # ambient only: 0.2 * cd


def test_mesh_without_triangles_is_empty_tree():
    rs = RawScene([{"kind": "mesh", "positions": np.zeros((0, 3)), "indices": []},
                   {"kind": "plane", "point": (0, 0, 2), "normal": (0, 0, -1), "tangent": (1, 0, 0)}],
                  [{"kind": "diffuse"}], [{"kind": "point", "vec": (0, 1, 0), "color": (5, 5, 5), "radius": 1.0}])
    both(rs, 32, 24)


def test_all_material_kinds_and_transparent_recursion():
    mats = [{"kind": "diffuse", "color1": (0.9, 0.2, 0.2)}, {"kind": "plastic", "ior": 1.9, "color1": (0.2, 0.9, 0.2)},
            {"kind": "mirror", "ior": 4.0}, {"kind": "emmit", "color1": (3, 2, 1)}, {"kind": "transparent", "ior": 1.5},
            {"kind": "shownormal"}, {"kind": "showuv"},
            {"kind": "plastic", "ior": 1.3, "cmap": "checker", "color1": (1, 1, 1), "color2": (0.1, 0.1, 0.1), "size": 0.4}]
    objs = [{"kind": "sphere", "center": (-1.5 + 0.75 * i, 0.2 * (i % 2), 0.5), "radius": 0.33, "material": i} for i in range(7)]
    objs += [{"kind": "sphere", "center": (0.0, 0.9, 0.0), "radius": 0.4, "material": 4},    # transparent in front of transparent
             {"kind": "plane", "point": (0, -0.6, 0), "normal": (0, 1, 0), "tangent": (1, 0, 0), "material": 7},
             {"kind": "plane", "point": (0, 0, 3), "normal": (0, 0, -1), "tangent": (1, 0, 0), "material": 0},
             dict(kind="mesh", material=1, **grid_mesh(8, z=1.5, wobble=0.05))]
    lights = [{"kind": "point", "vec": (0, 2, -1), "color": (20, 20, 20), "radius": 0.5},
              {"kind": "directional", "vec": (0.3, -1, 0.5), "color": (0.6, 0.6, 0.7)}]
    rs = RawScene(objs, mats, lights, camera={"position": (0, 0.3, -3), "target": (0, 0, 0.5)})
    for depth in (0, 1, 3, 5):
        img, ref = both(rs, 160, 120, depth=depth)
    assert ref["rays"]["probe"] > 0 and ref["rays"]["exit"] > 0 and ref["rays"]["reflect"] > 0


def test_orthographic_camera_and_uv_mesh_texture():
    tex = np.random.RandomState(3).uniform(0, 1, size=(5, 7, 3))
    mats = [{"kind": "diffuse", "cmap": "texture", "texture": 0}, {"kind": "plastic", "cmap": "texture", "texture": 0, "ior": 1.5}]
    objs = [dict(kind="mesh", material=0, **grid_mesh(6, z=0.3, wobble=0.1)),
            {"kind": "sphere", "center": (0, 0, -0.5), "radius": 0.5, "material": 1}]
    lights = [{"kind": "directional", "vec": (0.2, 0.3, 1.0), "color": (1.5, 1.5, 1.5)}]
    # Projection.hs:30-32: the orthographic view plane is in PIXEL units, so keep the scene pixel-sized
    for o in objs:
        if o["kind"] == "mesh":
            o["positions"] = np.asarray(o["positions"]) * 30
        else:
            o["center"] = tuple(30 * c for c in o["center"])
            o["radius"] *= 30
    rs = RawScene(objs, mats, lights, textures=[tex],
                  camera={"position": (3, 2, -80), "target": (0, 0, 0), "projection": "orthographic"})
    both(rs, 96, 64)


def test_more_than_32_lights_uses_the_simple_shadow_kernel():
    rng = np.random.RandomState(5)
    lights = [{"kind": "point", "vec": tuple(rng.uniform(-1, 1, 3) * (1.5, 0.5, 1.5) + (0, 1.5, 0)), "color": (0.4, 0.4, 0.4),
               "radius": 0.5} for _ in range(40)]
    objs = [{"kind": "plane", "point": (0, -0.5, 0), "normal": (0, 1, 0), "tangent": (1, 0, 0)},
            dict(kind="mesh", material=0, **grid_mesh(5, z=0.0, wobble=0.2)),
            {"kind": "sphere", "center": (0.5, 0, 0), "radius": 0.3}]
    rs = RawScene(objs, [{"kind": "diffuse", "color1": (0.8, 0.8, 0.8)}], lights, camera={"position": (0, 1, -3)})
    both(rs, 80, 60)


def test_more_than_64_objects_reads_tables_from_global_memory():
    rng = np.random.RandomState(9)
    mats = [{"kind": k, "ior": 1.5, "color1": tuple(rng.uniform(0.2, 1, 3))} for k in ("diffuse", "plastic", "mirror")] * 30
    objs = [{"kind": "sphere", "center": tuple(rng.uniform(-1, 1, 3)), "radius": float(rng.uniform(0.03, 0.12)), "material": i % 90}
            for i in range(150)]
    objs.append({"kind": "plane", "point": (0, -1.2, 0), "normal": (0, 1, 0), "tangent": (1, 0, 0), "material": 0})
    lights = [{"kind": "point", "vec": (0, 3, -2), "color": (60, 60, 60), "radius": 0.5}]
    rs = RawScene(objs, mats, lights, camera={"position": (0, 0, -4)})
    both(rs, 120, 90)


def test_sphere_tree_ties_emitters_and_interleaved_objects():
    """>= 16 top-level spheres are walked through the sphere tree (any order): coincident spheres must resolve to the
    lowest object index (RayHs.hs:67-71), emitter spheres must not occlude (RayHs.hs:81-82), and planes / meshes placed
    between the spheres in the object list keep their place in the tie order.  The exact-box walk (all spheres, like the
    reference's scan) must give the same image."""
    rng = np.random.RandomState(11)
    mats = [{"kind": "diffuse", "color1": (0.9, 0.3, 0.2)}, {"kind": "plastic", "ior": 1.7, "color1": (0.2, 0.8, 0.3)},
            {"kind": "mirror", "ior": 3.0}, {"kind": "emmit", "color1": (2, 2, 1)}, {"kind": "transparent", "ior": 1.4},
            {"kind": "diffuse", "color1": (0.2, 0.3, 0.9)}]
    objs = []
    for i in range(60):
        c = tuple(rng.uniform(-1.2, 1.2, 3) * (1, 0.7, 1))
        r = float(rng.uniform(0.05, 0.25))
        objs.append({"kind": "sphere", "center": c, "radius": r, "material": i % 5})
        if i % 7 == 0:   # an identical sphere later in the list with another material: never visible
            objs.append({"kind": "sphere", "center": c, "radius": r, "material": 5})
        if i == 10:
            objs.append({"kind": "plane", "point": (0, -0.9, 0), "normal": (0, 1, 0), "tangent": (1, 0, 0), "material": 1})
        if i == 30:
            objs.append(dict(kind="mesh", material=0, **grid_mesh(6, z=1.6, wobble=0.1)))
    # a sphere tangent to the floor plane and one centred on a light (emitter): shadow-rule edge cases
    objs.append({"kind": "sphere", "center": (0.3, -0.7, -0.4), "radius": 0.2, "material": 0})
    objs.append({"kind": "sphere", "center": (0.0, 1.6, -0.5), "radius": 0.15, "material": 3})
    lights = [{"kind": "point", "vec": (0.0, 1.6, -0.5), "color": (25, 25, 25), "radius": 0.5},
              {"kind": "directional", "vec": (-0.4, 1.0, -0.6), "color": (0.5, 0.5, 0.6)}]
    rs = RawScene(objs, mats, lights, camera={"position": (0, 0.4, -3.5), "target": (0, 0, 0)})
    img, ref = both(rs, 161, 121)
    assert ref["rays"]["probe"] > 0 and ref["rays"]["reflect"] > 0
    img2, _ = both(rs, 161, 121, exact_boxes=True)
    assert np.array_equal(img.pixels, img2.pixels)
    assert not (img.hit_ids[..., 0] >= 0).all() and (img.hit_ids[..., 0] >= 0).any()
    ids = set(np.unique(img.hit_ids[..., 0]).tolist())
    dup = [k for k, o in enumerate(objs) if o.get("material") == 5]
    assert not ids.intersection(dup), "a coincident later sphere won a tie"


def test_synthetic_stress_scene_sphere_tree_and_spp():
    """configs[4] shape at reduced size with enough spheres for the sphere tree, 4 spp, hit ids and ray counts."""
    sc = rh.Scene.synthetic(60000, 300)
    w, h, spp = 160, 90, 4
    off = rh.sample_offsets(w * h, spp, 24)
    job = rh.renderingFromScene(sc, w, h)
    img = render_linear(job, spp=spp, offsets=off)
    ref = OracleScene(sc.raw).render(sc.camera, w, h, sc.max_depth, spp=spp, offsets=off)
    assert np.array_equal(img.hit_ids.reshape(h, w, spp, 2), ref["hit_ids"])
    print("straddled channels", assert_oracle_exact(img.pixels, img.linear, ref))
    got = tuple(img.stats[k] for k in ("rays_primary", "rays_reflect", "rays_probe", "rays_exit", "rays_shadow"))
    assert got == tuple(ref["rays"][k] for k in ("primary", "reflect", "probe", "exit", "shadow"))


def test_synthetic_stress_scene_small():
    """BASELINE.json configs[4] at reduced size: random triangles + spheres + checker floor, dragon.json camera/lights."""
    sc = rh.Scene.synthetic(30000, 40)
    w, h = 192, 108
    job = rh.renderingFromScene(sc, w, h)
    img = render_linear(job)
    ref = OracleScene(sc.raw).render(sc.camera, w, h, sc.max_depth)
    assert np.array_equal(img.hit_ids.reshape(h, w, 2), ref["hit_ids"].reshape(h, w, 2))
    print("straddled channels", assert_oracle_exact(img.pixels, img.linear, ref))


def test_centre_row_and_column_rays_take_the_exact_path():
    """Rays with a zero direction component (App. A-N1): cube faces at the camera's x and y, NaN slab arithmetic."""
    c = dict(positions=[(0, 0, 0), (1, 0, 0), (1, 1, 0), (0, 1, 0), (0, 0, 1), (1, 0, 1), (1, 1, 1), (0, 1, 1)],
             indices=[0, 1, 2, 0, 2, 3, 4, 6, 5, 4, 7, 6, 0, 4, 5, 0, 5, 1, 3, 2, 6, 3, 6, 7, 0, 3, 7, 0, 7, 4, 1, 5, 6, 1, 6, 2])
    g = grid_mesh(6, z=2.0)   # vertices on x = 0 and y = 0 lines, splits land exactly on the centre ray
    rs = RawScene([dict(kind="mesh", material=0, **c), dict(kind="mesh", material=0, **g)], [{"kind": "diffuse"}],
                  [{"kind": "point", "vec": (0, 0, -1), "color": (3, 3, 3), "radius": 1.0}])
    both(rs, 64, 64)
    both(rs, 65, 63)


def test_scene_far_from_the_coordinate_origin_keeps_parity_and_the_float_cull():
    """The float cull boxes are stored relative to the middle of the scene: a scene translated by (1e6, -2e6, 3e6) must
    still match its oracle bit for bit AND still cull (node visits within 2x of the untranslated scene; absolute float
    coordinates would resolve nothing at 1e6 and every ray would visit the whole tree)."""
    def scene(shift):
        sx, sy, sz = shift
        g = grid_mesh(24, z=1.0, wobble=0.15)
        g["positions"] = np.asarray(g["positions"]) + np.array(shift)
        objs = [dict(kind="mesh", material=1, **g),
                {"kind": "sphere", "center": (sx + 0.4, sy - 0.2, sz + 0.3), "radius": 0.3, "material": 0},
                {"kind": "plane", "point": (sx, sy - 0.8, sz), "normal": (0, 1, 0), "tangent": (1, 0, 0), "material": 0}]
        mats = [{"kind": "diffuse", "color1": (0.8, 0.7, 0.6)}, {"kind": "plastic", "ior": 1.6, "color1": (0.3, 0.6, 0.9)}]
        lights = [{"kind": "point", "vec": (sx + 0.5, sy + 1.5, sz - 1.0), "color": (30, 30, 30), "radius": 0.5}]
        return RawScene(objs, mats, lights, camera={"position": (sx, sy + 0.3, sz - 2.5), "target": (sx, sy, sz + 0.5)})

    near, far = scene((0.0, 0.0, 0.0)), scene((1e6, -2e6, 3e6))
    both(near, 160, 120)
    both(far, 160, 120)
    job_n, job_f = rh.Rendering(near, near.camera, 160, 120, 3), rh.Rendering(far, far.camera, 160, 120, 3)
    n = rh.render(job_n, count=True, shadow="pooled").stats
    f = rh.render(job_f, count=True, shadow="pooled").stats
    assert f["node_visits"] + f["shadow_node_visits"] < 2 * (n["node_visits"] + n["shadow_node_visits"]), (n, f)


def test_scene_beyond_the_shared_memory_occluder_tables():
    """14 lights, 18 occluding planes and 9 meshes exceed the shared-memory occluder tables (12 / 16 / 8): the light fold
    reads the occluder records from global memory and walks whenever there is a tree; same image."""
    rng = np.random.RandomState(21)
    lights = [{"kind": "point", "vec": tuple(rng.uniform(-1, 1, 3) * (1.2, 0.3, 1.2) + (0, 1.6, 0.3)), "color": (1.5, 1.5, 1.5),
               "radius": 0.5} for _ in range(13)] + [{"kind": "directional", "vec": (0.2, 1.0, -0.3), "color": (0.2, 0.2, 0.2)}]
    objs = [{"kind": "plane", "point": (0, -0.6, 0), "normal": (0, 1, 0), "tangent": (1, 0, 0), "material": 0}]
    for k in range(17):   # slanted planes behind and beside the scene
        a = 0.37 * k
        objs.append({"kind": "plane", "point": (3 * np.cos(a), 0, 2.5 + 3 * abs(np.sin(a))), "normal": (-np.cos(a), 0.1, -abs(np.sin(a)) - 0.2),
                     "tangent": (0, 1, 0), "material": k % 2})
    for k in range(9):
        g = grid_mesh(5, z=0.6 + 0.15 * k, wobble=0.05, seed=k)
        g["positions"] = np.asarray(g["positions"]) * 0.25 + np.array([-1 + 0.25 * k, -0.2 + 0.05 * k, 0])
        objs.append(dict(kind="mesh", material=k % 2, **g))
    mats = [{"kind": "diffuse", "color1": (0.7, 0.7, 0.6)}, {"kind": "plastic", "ior": 1.5, "color1": (0.4, 0.6, 0.8)}]
    rs = RawScene(objs, mats, lights, camera={"position": (0, 0.5, -3), "target": (0, 0, 1)})
    both(rs, 120, 90)


def test_eleven_lights_fit_the_fast_shadow_kernels():
    """11 lights: the most the fast shadow kernels take with one hit per lane per batch (pair terms in shared memory)."""
    rng = np.random.RandomState(33)
    lights = [{"kind": "point", "vec": tuple(rng.uniform(-1, 1, 3) * (1.5, 0.4, 1.5) + (0, 1.4, 0.2)), "color": (2.0, 1.8, 1.6),
               "radius": 0.4} for _ in range(11)]
    objs = [{"kind": "plane", "point": (0, -0.5, 0), "normal": (0, 1, 0), "tangent": (1, 0, 0), "material": 0},
            dict(kind="mesh", material=1, **grid_mesh(10, z=0.8, wobble=0.2)),
            {"kind": "sphere", "center": (-0.4, -0.1, 0.2), "radius": 0.35, "material": 1}]
    mats = [{"kind": "diffuse", "color1": (0.8, 0.8, 0.7)}, {"kind": "plastic", "ior": 1.7, "color1": (0.5, 0.7, 0.4)}]
    rs = RawScene(objs, mats, lights, camera={"position": (0, 0.6, -3), "target": (0, 0, 0.5)})
    both(rs, 150, 100)


def test_planes_that_shadow_from_either_side():
    """Occluder planes between the shaded points and the lights: a slanted shelf with a non-unit normal, a back wall a light
    sits behind, point lights on both sides of the shelf (one almost in its plane), a directional light that grazes the
    floor and one that is parallel to the shelf.  The shadow kernels decide most (pair, plane) cases from which side of
    the plane the ray starts (stage_plane_sides); the image must still be the oracle's, byte for byte."""
    lights = [{"kind": "point", "vec": (0.3, 1.6, 0.4), "color": (2.0, 1.9, 1.8), "radius": 0.6},     # above the shelf
              {"kind": "point", "vec": (-0.8, 0.2, -0.2), "color": (1.2, 1.4, 1.6), "radius": 0.5},   # below it
              {"kind": "point", "vec": (0.5, 0.9 + 1e-7, 0.5), "color": (1.0, 1.0, 1.0), "radius": 0.3},  # (almost) in its plane
              {"kind": "point", "vec": (0.0, 0.4, 3.5), "color": (1.5, 1.5, 1.5), "radius": 0.8},     # behind the back wall
              {"kind": "directional", "vec": (0.6, 1e-4, -0.3), "color": (0.5, 0.4, 0.3)},            # grazes the floor
              {"kind": "directional", "vec": (2.0, 0.4, 0.0), "color": (0.3, 0.4, 0.5)}]              # parallel to the shelf
    objs = [{"kind": "plane", "point": (0, -0.6, 0), "normal": (0, 1, 0), "tangent": (1, 0, 0), "material": 0},
            {"kind": "plane", "point": (0.5, 0.9, 0.5), "normal": (-0.6, 3.0, 0.0), "tangent": (1, 0.2, 0), "material": 1},  # the shelf
            {"kind": "plane", "point": (0, 0, 3.0), "normal": (0, 0, -1), "tangent": (1, 0, 0), "material": 0},
            {"kind": "sphere", "center": (-0.3, -0.2, 0.6), "radius": 0.4, "material": 1},
            {"kind": "sphere", "center": (0.7, 1.3, 0.9), "radius": 0.25, "material": 0},
            dict(kind="mesh", material=1, **grid_mesh(6, z=1.4, wobble=0.15))]
    mats = [{"kind": "diffuse", "color1": (0.8, 0.8, 0.7)}, {"kind": "plastic", "ior": 1.6, "color1": (0.5, 0.6, 0.8)}]
    rs = RawScene(objs, mats, lights, camera={"position": (0.2, 0.3, -3.2), "target": (0, 0.3, 1)})
    img, ref = both(rs, 200, 150)
    assert np.array_equal(img.pixels, ref["rgb_u8"])
    rs2 = RawScene(objs, mats, lights, camera={"position": (0.2, 1.8, -2.0), "target": (0, 0.5, 1)})  # from above the shelf
    img2, ref2 = both(rs2, 160, 120)
    assert np.array_equal(img2.pixels, ref2["rgb_u8"])
