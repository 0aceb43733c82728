"""The kernels switch code paths at table-size limits: shared-memory object / material / light tables, the staged occluder
tables and light masks of the fast shadow kernels, the per-lane-refill schedule's root stack, the sphere tree, the cube
maps' resolution, the packed lit-triangle flags and map index, the deep traversal stack, the pass count of the deepest
ray tree, and the warp, batch and slab edges of the queues.  Each rung below is two or three hand-built scenes, equal
but for the entries that move one limit, on either side of it.  Every scene asserts the side it is on, and every render
of it — pooled and per-lane-refill shadow walks, light maps off, the exact box walk; one sample at the pixel and three
seeded ones — is held to the oracle channel by channel (tests/util.py assert_oracle_exact), hit ids and ray counts
exactly; without a Transparent material the variants agree bit for bit.  Where a rung adds a light or an occluder, the
oracle's image must change at >= 1 % of its pixels, and the added light or occluder must shadow some of them, so that
the side that crosses the limit really exercises the path it selects."""
import ctypes as C

import numpy as np
import pytest

import rayhs_b200 as rh
from oracle.orc import OracleScene
from rayhs_b200 import capi
from tests.util import RawScene, assert_oracle_exact, render_linear

pytestmark = pytest.mark.gpu

W, H = 96, 72
SEED = 41
SAMPLES = ((1, None), (3, SEED))   # one sample at each pixel; three of sample_offsets(W * H, 3, SEED)
VARIANTS = {"pooled": dict(shadow="pooled"), "split": dict(shadow="split"), "no maps": dict(light_maps=False),
            "exact boxes": dict(exact_boxes=True)}
COUNTS = ("primary", "reflect", "probe", "exit", "shadow")
CAMERA = {"position": (0.0, 1.6, -4.2), "target": (0.0, -0.4, 0.8)}
GREY = {"kind": "diffuse", "color1": (0.75, 0.75, 0.7)}
BLUE = {"kind": "plastic", "ior": 1.5, "color1": (0.3, 0.5, 0.9)}


# ---------------------------------------------------------------------------------------------------- scene pieces
def floor(material=0):
    return {"kind": "plane", "point": (0, -1, 0), "normal": (0, 1, 0), "tangent": (1, 0, 0), "material": material}


def sphere(c, r, material=1):
    return {"kind": "sphere", "center": tuple(float(x) for x in c), "radius": float(r), "material": material}


def tile(center, u, v, n=2, material=1):
    """A flat parallelogram mesh center + s u + t v (s, t in [-1, 1]) of 2 n^2 triangles, normals along v x u."""
    center, u, v = (np.asarray(x, dtype=np.float64) for x in (center, u, v))
    nrm = np.cross(v, u)
    nrm /= np.linalg.norm(nrm)
    s = np.linspace(-1, 1, n + 1)
    pos = np.array([center + a * u + b * v for b in s for a in s])
    idx = []
    for j in range(n):
        for i in range(n):
            a = j * (n + 1) + i
            idx += [a, a + 1, a + n + 2, a, a + n + 2, a + n + 1]
    uv = np.array([((a + 1) / 2, (b + 1) / 2) for b in s for a in s])
    return {"kind": "mesh", "material": material, "positions": pos, "normals": np.tile(nrm, (len(pos), 1)), "uvs": uv,
            "indices": idx}


def point(p, c=1.0, radius=2.0):
    return {"kind": "point", "vec": tuple(float(x) for x in p), "color": (c, c, c), "radius": radius}


def ring_lights(n, c, height=2.6, r=2.4, z=0.6):
    """n point lights on a circle above the scene, in an order that spreads consecutive ones around it."""
    return [point((r * np.cos(2.399963 * k), height + 0.15 * (k % 3), z + r * np.sin(2.399963 * k)), c) for k in range(n)]


class Side:
    """One scene of a rung: its objects, materials and lights (kept for the shadow probe), the RawScene, and the
    assertion of the side of the limit it is on (check(side) -> printable evidence)."""

    def __init__(self, label, objects, materials, lights, check, max_depth=3, camera=CAMERA, frames=((W, H, SAMPLES),)):
        self.label, self.objects, self.materials, self.lights = label, objects, materials, lights
        self.check, self.max_depth, self.frames = check, max_depth, frames
        self.rs = RawScene(objects, materials, lights, camera=camera, size=(W, H, max_depth))


def info4(side):
    """rh_scene_info: [tables_in_smem, shadow_fast, max tree depth, deep-stack entries]."""
    info = (C.c_int32 * 4)()
    capi.check(capi.lib().rh_scene_info(side.rs.device, None, info))
    return list(info)


def tables(side):
    return rh.Scene.light_tables(side.rs)   # (RawScene offers the views these methods read: device, flat)


def stats(side, **kw):
    return rh.render(rh.Rendering(side.rs, side.rs.camera, W, H, side.max_depth), **kw).stats


def expect_info(smem, fast):
    def check(side):
        got = info4(side)
        assert got[:2] == [smem, fast], (side.label, "info4", got)
        return {"info4": got}
    return check


def expect_split(smem, fast, split):
    """The forced per-lane-refill schedule runs (shadow_split 1) or is refused for this scene (0: pooled)."""
    def check(side):
        got = info4(side)
        assert got[:2] == [smem, fast], (side.label, "info4", got)
        s = stats(side, shadow="split")["shadow_split"]
        assert s == split, (side.label, "shadow_split", s)
        return {"info4": got, "shadow_split": s}
    return check


# ---------------------------------------------------------------------------------------------------- the rungs
def rung_objects():
    """64 | 65 objects (the floor and 63 | 64 spheres): the object table is staged in shared memory up to 64.  The spheres
    are walked through the sphere tree, so the occluder tables stay within the fast shadow kernels' on both sides."""
    xs, zs = np.linspace(-2.2, 2.2, 9), np.linspace(-0.2, 3.0, 7)
    balls = [sphere((x, -0.86, z), 0.14, 1 + (i % 2)) for i, (z, x) in enumerate((z, x) for z in zs for x in xs)]
    added = sphere((0.5, -0.45, -0.9), 0.55, 2)
    mats = [GREY, BLUE, {"kind": "diffuse", "color1": (0.9, 0.4, 0.3)}]
    lights = [point((-1.5, 2.8, -1.8), 9.0), point((1.8, 1.2, -1.2), 5.0)]
    return [Side("64 objects", [floor()] + balls, mats, lights, expect_info(1, 1)),
            Side("65 objects", [floor()] + balls + [added], mats, lights, expect_info(0, 1))], ("object", 64)


def rung_materials():
    """64 | 65 materials: the material table is staged in shared memory up to 64.  The objects read materials from all
    over the table; the large front sphere takes material 0 on one side and the added material 64 on the other."""
    mats = [{"kind": ("diffuse", "plastic")[k % 2], "ior": 1.3 + 0.01 * k,
             "color1": (0.3 + 0.01 * k, 0.9 - 0.01 * k, 0.5 + 0.005 * k)} for k in range(64)]
    objs = [floor(63)] + [sphere((-2.0 + 0.45 * k, -0.8, 1.5 + 0.3 * (k % 3)), 0.2, (5 * k + 7) % 64) for k in range(10)]
    lights = [point((-1.2, 2.6, -1.5), 9.0), point((2.0, 1.5, 0.0), 4.0)]
    front = dict(sphere((0.3, -0.4, -0.6), 0.6, 0))
    other = dict(front, material=64)
    red = {"kind": "plastic", "ior": 1.9, "color1": (0.95, 0.1, 0.1)}
    return [Side("64 materials", objs + [front], mats, lights, expect_info(1, 1)),
            Side("65 materials", objs + [other], mats + [red], lights, expect_info(0, 1))], ("material", 64)


def lit_scene(lights, mats=(GREY, BLUE)):
    objs = [floor(), tile((0.0, 0.1, 0.8), (0.9, 0.0, 0.0), (0.0, 0.25, 0.6), n=4),
            sphere((-1.2, -0.5, 0.0), 0.5), sphere((1.3, -0.6, -0.2), 0.4, 0), sphere((0.2, -0.75, -1.0), 0.25)]
    return objs, list(mats), lights


def rung_smem_lights():
    """16 | 17 lights: the light table is staged in shared memory up to 16 (both sides are beyond the fast shadow
    kernels' 12)."""
    base = ring_lights(16, 0.9)
    added = point((-2.2, 0.6, -1.6), 6.0)
    return [Side("16 lights", *lit_scene(base), expect_info(1, 0)),
            Side("17 lights", *lit_scene(base + [added]), expect_info(0, 0))], ("light", 16)


def rung_fast_lights():
    """12 | 13 lights: the fast shadow kernels (staged occluder tables, per-light masks of plane and root-box sides,
    cube maps, lit flags) take up to 12 lights."""
    base = ring_lights(12, 1.1)
    added = point((-2.2, 0.6, -1.6), 6.0)
    return [Side("12 lights", *lit_scene(base), expect_info(1, 1)),
            Side("13 lights", *lit_scene(base + [added]), expect_info(1, 0))], ("light", 12)


def rung_planes():
    """16 | 17 occluding planes, and 17 planes of which one is Emmit (16 occluders: still fast).  Fourteen planes stand
    behind the camera facing the scene; the added one is a wall between the scene and the second light."""
    behind = [{"kind": "plane", "point": (0, 0, -6.0 - 0.3 * k), "normal": (0.04 * k - 0.28, 0.02 * k - 0.1, 1.0),
               "tangent": (1, 0, 0), "material": k % 2} for k in range(14)]
    back = {"kind": "plane", "point": (0, 0, 4.0), "normal": (0, 0, -1), "tangent": (1, 0, 0), "material": 0}
    objs = [floor(), back] + behind + [sphere((-0.6, -0.55, 0.6), 0.45), sphere((0.4, -0.8, -0.8), 0.2, 0)]
    wall = {"kind": "plane", "point": (1.3, 0, 0), "normal": (-1.0, 0.0, 0.25), "tangent": (0, 1, 0), "material": 1}
    mats = [GREY, BLUE, {"kind": "emmit", "color1": (0.4, 0.3, 0.2)}]
    lights = [point((-1.5, 2.6, -1.5), 7.0), point((3.2, 1.8, 1.0), 9.0)]
    return [Side("16 planes", objs, mats, lights, expect_info(1, 1)),
            Side("17 planes", objs + [wall], mats, lights, expect_info(1, 0)),
            Side("17 planes, one Emmit", objs + [dict(wall, material=2)], mats, lights, expect_info(1, 1))], ("object", 18)


def rung_meshes():
    """8 | 9 occluder meshes: the fast shadow kernels stage up to 8 mesh roots."""
    meshes = [tile((-2.0 + 0.55 * k, -0.2 + 0.12 * (k % 3), 1.6 + 0.35 * (k % 2)), (0.22, 0.0, 0.05), (0.0, 0.2, 0.1), n=3)
              for k in range(8)]
    added = tile((0.2, 0.2, -0.3), (0.5, 0.0, 0.1), (0.0, 0.05, 0.45), n=3, material=0)
    objs = [floor(), sphere((0.9, -0.6, 0.4), 0.4)]
    lights = [point((-1.0, 2.8, -1.6), 9.0), point((1.5, 2.0, -0.5), 5.0)]
    return [Side("8 meshes", objs + meshes, [GREY, BLUE], lights, expect_info(1, 1)),
            Side("9 meshes", objs + meshes + [added], [GREY, BLUE], lights, expect_info(1, 0))], ("object", 10)


def expect_spheres(fast, tree):
    """shadow_fast, and whether the spheres are walked through the sphere tree: the scene has no mesh, so only the
    sphere tree makes node visits."""
    def check(side):
        got = info4(side)
        visits = stats(side, count=True)["node_visits"]
        assert got[1] == fast and got[0] == 1, (side.label, "info4", got)
        assert (visits > 0) == tree, (side.label, "node_visits", visits)
        return {"info4": got, "node_visits": visits}
    return check


def rung_spheres():
    """15 linear spheres | 16 (the sphere tree) | 17 of which one is centred at x = 1e30, out of view: the tree is
    refused (a centre coordinate or radius >= 1e30 or NaN), and 17 linear occluder spheres exceed the fast shadow
    kernels' 16.  That is the only way to get more than 16 linear occluder spheres: with the tree, spheres are not in
    the occluder tables at all, so the sphere clause of shadow_fast matters only for such scenes."""
    balls = [sphere((-2.0 + 0.3 * k, -0.8 + 0.02 * k, 1.2 + 0.4 * (k % 4)), 0.17, k % 2) for k in range(15)]
    added = sphere((0.2, -0.4, -0.7), 0.55)
    far = sphere((1e30, 0.0, 0.0), 1.0)
    lights = [point((-1.3, 2.7, -1.7), 9.0), point((1.8, 1.6, -0.8), 5.0)]
    objs = [floor()] + balls
    return [Side("15 spheres", objs, [GREY, BLUE], lights, expect_spheres(1, False)),
            Side("16 spheres", objs + [added], [GREY, BLUE], lights, expect_spheres(1, True)),
            Side("17 spheres, one at 1e30", objs + [added, far], [GREY, BLUE], lights, expect_spheres(0, False))], ("object", 16)


def rung_mask_lights():
    """32 | 33 lights: the per-lane-refill schedule keeps a hit's lights in 32-bit walk / settled masks; beyond 32 the
    forced schedule falls back to pooled."""
    base = ring_lights(32, 0.45)
    added = point((-2.2, 0.6, -1.6), 6.0)
    return [Side("32 lights", *lit_scene(base), expect_split(0, 0, 1)),
            Side("33 lights", *lit_scene(base + [added]), expect_split(0, 0, 0))], ("light", 32)


def rung_roots():
    """64 | 65 occluder roots: the per-lane-refill schedule stacks every tree root of the scene and is possible up to 64.
    The floor is a mesh too and there are no spheres (no sphere-tree root); 64 | 65 meshes are also 64 | 65 objects, so
    the shared-memory object table's limit is crossed at the same step — no scene separates the two."""
    ground = tile((0.0, -1.0, 2.0), (6.0, 0.0, 0.0), (0.0, 0.0, 6.0), n=2, material=0)
    xs, zs = np.linspace(-2.4, 2.4, 9), np.linspace(0.0, 3.5, 7)
    posts = [tile((x, -0.75, z), (0.12, 0.0, 0.0), (0.0, 0.22, 0.05), n=1, material=1 + (i % 2))
             for i, (z, x) in enumerate((z, x) for z in zs for x in xs)]
    added = tile((0.3, -0.3, -0.8), (0.5, 0.0, 0.1), (0.0, 0.4, 0.2), n=2, material=1)
    mats = [GREY, BLUE, {"kind": "diffuse", "color1": (0.9, 0.4, 0.3)}]
    lights = [point((-1.4, 2.8, -1.9), 9.0), point((1.8, 1.3, -1.4), 5.0)]
    return [Side("64 roots", [ground] + posts, mats, lights, expect_split(1, 0, 1)),
            Side("65 roots", [ground] + posts + [added], mats, lights, expect_split(0, 0, 0))], ("object", 64)


def map_meshes(n):
    return [tile((-2.0 + 0.8 * k, -0.3 + 0.15 * (k % 2), 1.0 + 0.5 * (k % 3)), (0.3, 0.0, 0.05), (0.0, 0.25, 0.15), n=3)
            for k in range(n)]


def expect_res(res):
    def check(side):
        got, t = info4(side), tables(side)
        assert got[:2] == [1, 1], (side.label, "info4", got)
        assert t["res"] == res, (side.label, "res", t["res"])
        assert len(t["maps"]) > 0 and t["lit"] is not None, (side.label, "no maps or lit flags")
        return {"info4": got, "res": t["res"], "maps": len(t["maps"])}
    return check


def map_res_scene(n_point):
    """6 occluder meshes and n_point point lights (the cube maps are built for every (point light, mesh) pair)."""
    lights = [point((-2.4 + 0.75 * k, 2.2 + 0.3 * (k % 2), -1.5 + 0.4 * (k % 3)), 2.2) for k in range(7)]
    lights += [point((1.6, 1.4, -1.8), 6.0)][: n_point - 7]
    return [floor(), sphere((0.9, -0.65, -0.4), 0.35)] + map_meshes(6), [GREY, BLUE], lights


def rung_map_res():
    """7 | 8 point lights x 6 meshes = 42 | 48 cube maps: the maps of a scene share a 256 MiB budget, 42 maps of 512^2
    cells per face fit and 43 do not, so the resolution halves to 256.  Maps exist only for scenes the fast shadow
    kernels take, at most 12 x 8 = 96 pairs, so the resolutions 128 and 64 the halving allows never occur."""
    return [Side("42 maps", *map_res_scene(7), expect_res(512)),
            Side("48 maps", *map_res_scene(8), expect_res(256))], ("light", 7)


def packed_scene(n_lights):
    """8 occluder meshes; 4 directional lights first, then point lights, so that a light's index (the lit bit and the
    map index light * 8 + mesh) is not its index among the point lights."""
    dirs = [{"kind": "directional", "vec": v, "color": (0.12, 0.12, 0.12)}
            for v in ((0.3, 1.0, -0.4), (-0.5, 1.0, -0.2), (0.1, 1.0, 0.6), (-0.2, 0.8, -0.9))]
    pts = [point((-2.4 + 0.8 * k, 2.3 + 0.2 * (k % 2), -1.2 + 0.3 * (k % 3)), 1.6) for k in range(7)]
    pts += [point((1.04, -0.23, -2.04), 5.0)]   # light 11: in front of mesh 7, which shadows mesh 3 and the floor from it
    meshes = map_meshes(7) + [tile((0.8, -0.2, -0.9), (0.35, 0.0, 0.0), (0.0, 0.3, 0.15), n=3)]
    return [floor(), sphere((-1.0, -0.7, -0.6), 0.3)] + meshes, [GREY, BLUE], (dirs + pts)[:n_lights]


def expect_packed(n_lights):
    def check(side):
        got, t = info4(side), tables(side)
        assert got[:2] == [1, 1], (side.label, "info4", got)
        lit, index = t["lit"], t["index"]
        assert lit is not None and index.shape == (n_lights, 8), (side.label, index.shape)
        last = n_lights - 1
        on_mesh7 = (lit >> 12) == 7
        bits = int(((lit[on_mesh7] >> last) & 1).sum())
        assert bits > 0, (side.label, f"no lit bits of light {last} on mesh 7")
        assert index[last, 7] != 0xFFFFFFFF, (side.label, f"no map for (light {last}, mesh 7)")
        assert (index[:4] == 0xFFFFFFFF).all(), (side.label, "a map for a directional light")
        return {"info4": got, "res": t["res"], f"lit bits of light {last} on mesh 7": bits,
                f"index[{last}, 7]": int(index[last, 7])}
    return check


def rung_packed():
    """11 | 12 lights x 8 meshes: the lit-triangle flags pack 12 light bits and the mesh index in bits 12-15, and the map
    index is light * 8 + mesh.  The added light 11 is the last bit and has a map and lit bits on mesh 7, the last index."""
    return [Side("11 lights x 8 meshes", *packed_scene(11), expect_packed(11)),
            Side("12 lights x 8 meshes", *packed_scene(12), expect_packed(12))], ("light", 11)


def tube(length, rings, around=6, r=0.05):
    """An open tube along +z from z = 0, rings x around quads, normals facing its axis."""
    a = np.linspace(0, 2 * np.pi, around, endpoint=False)
    zs = np.linspace(0.0, length, rings + 1)
    pos = np.array([(r * np.cos(t), r * np.sin(t), z) for z in zs for t in a])
    nrm = np.array([(-np.cos(t), -np.sin(t), 0.0) for z in zs for t in a])
    idx = []
    for j in range(rings):
        for i in range(around):
            p, q = j * around + i, j * around + (i + 1) % around
            idx += [p, q, q + around, p, q + around, p + around]
    return {"kind": "mesh", "material": 0, "positions": pos, "normals": nrm, "uvs": np.zeros((len(pos), 2)), "indices": idx}


def expect_pushes(deep):
    def check(side):
        got = info4(side)
        pushes = stats(side, count=True)["deep_stack_pushes"]
        assert (pushes > 0) == deep, (side.label, "deep_stack_pushes", pushes)
        return {"info4": got, "deep_stack_pushes": pushes}
    return check


def rung_deep_stack():
    """A thin tube 800 times as long as it is wide, of 48 000 triangles, seen down its axis from just outside its mouth:
    the tree splits it along its length, every box holds the axis, and a ray that travels far inside enters both
    children at every level, so its walk stacks more subtrees than the shared-memory short stack holds (8 entries) and
    goes on in the deep stack in global memory | a short one of the same rings (240 triangles): no walk leaves the short
    stack."""
    cam = {"position": (0.002, 0.001, -0.12), "target": (0.0, 0.0, 1.0)}
    lights = [point((0.0, 0.01, 0.1), 2.0, radius=0.2), point((0.01, 0.0, 3.0), 4.0, radius=0.5)]
    mats = [GREY]
    return [Side("short tube", [tube(0.2, 20)], mats, lights, expect_pushes(False), camera=cam),
            Side("long tube", [tube(40.0, 4000)], mats, lights, expect_pushes(True), camera=cam)], None


def expect_depth(depth):
    def check(side):
        st = stats(side, shadow="pooled")
        # most samples reach the deepest level: a reflection ray per level of every sample that never meets a sphere
        assert st["rays_reflect"] >= 0.5 * depth * W * H, (side.label, st["rays_reflect"])
        return {"max_depth": depth, "rays_reflect": st["rays_reflect"], "rays_probe": st["rays_probe"]}
    return check


def rung_depth():
    """max_depth 29 | 30 (the most rh_render accepts; 31 is refused) in a closed box of mirrors with a small diffuse and
    a small Transparent sphere: every path bounces to the last level, 2 * 30 + 1 = 61 passes of the 62 kMaxPasses allows
    when a Transparent hit forks a probe.  The Transparent sphere is small, so that a path meets it once or twice."""
    s = 1.5
    walls = [{"kind": "plane", "point": tuple(s * -n for n in nv), "normal": nv, "tangent": tv, "material": 0}
             for nv, tv in (((1, 0, 0), (0, 1, 0)), ((-1, 0, 0), (0, 1, 0)), ((0, 1, 0), (1, 0, 0)), ((0, -1, 0), (1, 0, 0)),
                            ((0, 0, 1), (1, 0, 0)), ((0, 0, -1), (1, 0, 0)))]
    objs = walls + [sphere((0.5, -0.6, 0.7), 0.3, 1), sphere((-0.6, 0.5, 0.9), 0.12, 2)]
    mats = [{"kind": "mirror", "ior": 6.0}, {"kind": "diffuse", "color1": (0.9, 0.6, 0.3)}, {"kind": "transparent", "ior": 1.4}]
    lights = [point((0.0, 1.2, -0.5), 20.0)]
    cam = {"position": (0.1, 0.2, -1.3), "target": (0.0, 0.0, 1.0)}
    return [Side("max_depth 29", objs, mats, lights, expect_depth(29), max_depth=29, camera=cam),
            Side("max_depth 30", objs, mats, lights, expect_depth(30), max_depth=30, camera=cam)], None


def rung_frame_size():
    """Frames of W * H * spp = 1, 31, 32, 33, 127, 128, 129 samples: the edges of a warp (32), of the queues' slabs (128)
    and of the resolve kernel's blocks (128), with one sample at the pixel or seeded samples."""
    frames = ((1, 1, ((1, None),)), (31, 1, ((1, None),)), (4, 8, ((1, None),)), (11, 1, ((3, SEED),)), (127, 1, ((1, None),)),
              (8, 8, ((2, SEED),)), (43, 1, ((3, SEED),)), (129, 1, ((1, None),)), (16, 8, ((1, None),)))
    objs, mats, lights = lit_scene([point((-1.2, 2.6, -1.5), 9.0), {"kind": "directional", "vec": (0.3, 1.0, -0.5), "color": (0.3,) * 3}])
    cam = {"position": (0.0, -0.55, -4.0), "target": (0.0, -2.6, 0.0)}   # row 0 (the view's top edge) crosses the spheres
    return [Side("frame sizes", objs, mats, lights, lambda side: {}, camera=cam, frames=frames)], None


RUNGS = {"objects": rung_objects, "materials": rung_materials, "smem_lights": rung_smem_lights, "fast_lights": rung_fast_lights,
         "planes": rung_planes, "meshes": rung_meshes, "spheres": rung_spheres, "mask_lights": rung_mask_lights,
         "roots": rung_roots, "map_res": rung_map_res, "packed_tables": rung_packed, "deep_stack": rung_deep_stack,
         "depth": rung_depth, "frame_size": rung_frame_size}


# ---------------------------------------------------------------------------------------------------- the checks
def has_transparent(side):
    return any(m["kind"] == "transparent" for m in side.materials)


def hold(side, w, h, spp, seed):
    """Renders every variant and holds each to the oracle; returns the oracle's render and the straddled channels."""
    job = rh.Rendering(side.rs, side.rs.camera, w, h, side.max_depth)
    offsets = rh.sample_offsets(w * h, spp, seed) if seed is not None else None
    ref = OracleScene(side.rs.raw).render(side.rs.camera, w, h, side.max_depth, spp=spp, offsets=offsets)
    want = tuple(ref["rays"][k] for k in COUNTS)
    first, straddled = None, {}
    for name, kw in VARIANTS.items():
        what = (side.label, (w, h, spp), name)
        img = render_linear(job, spp=spp, seed=seed, **kw)
        assert np.array_equal(img.hit_ids.reshape(h, w, spp, 2), ref["hit_ids"]), (what, "hit ids")
        got = tuple(img.stats["rays_" + k] for k in COUNTS)
        assert got == want, (what, got, want)
        straddled[name] = assert_oracle_exact(img.pixels, img.linear, ref, what)
        if first is None:
            first = img
        elif not has_transparent(side):
            assert np.array_equal(img.pixels, first.pixels), (what, "bytes differ from the pooled render")
            assert np.array_equal(img.linear.view(np.uint64), first.linear.view(np.uint64)), (what, "linear bits differ")
    return ref, straddled


def shadowed(side, light, by=None, step=2):
    """Camera pixels (every step-th row and column, through the pixel centre) whose first hit faces `light` and is
    shadowed from it — by object `by` if given — according to the oracle's closest-hit query."""
    orc = OracleScene(side.rs.raw)
    L = side.lights[light]
    n = 0
    for py in range(0, H, step):
        for px in range(0, W, step):
            o, d = orc.ray_from_pixel(side.rs.camera, W, H, px + 0.5, py + 0.5)
            hit = orc.closest(o, d)
            if hit is None:
                continue
            p = hit["p"]
            ld = np.asarray(L["vec"], dtype=np.float64) - (p if L["kind"] == "point" else 0)
            dist = np.linalg.norm(ld) if L["kind"] == "point" else np.inf
            ld = ld / np.linalg.norm(ld)
            if np.dot(ld, hit["n"]) <= 0:
                continue
            o2 = p + 1e-6 * ld
            s = orc.closest(o2, ld)
            if s is None or np.linalg.norm(s["p"] - o2) >= dist:
                continue
            if side.materials[side.objects[s["object"]]["material"]]["kind"] == "emmit":
                continue
            n += by is None or s["object"] == by
    return n


@pytest.mark.parametrize("rung", list(RUNGS))
def test_limit_rung(rung):
    sides, added = RUNGS[rung]()
    images = []
    try:
        for side in sides:
            evidence = side.check(side)
            for (w, h, samples) in side.frames:
                for spp, seed in samples:
                    ref, straddled = hold(side, w, h, spp, seed)
                    if spp == 1 and (w, h) == (W, H):
                        images.append(ref["rgb_u8"])
                    print(rung, side.label, (w, h, spp), evidence, "rays", ref["rays"], "straddled", straddled)
        if added is not None:
            kind, index = added
            changed = (images[1] != images[0]).any(axis=-1).mean()
            assert changed >= 0.01, (rung, f"the added {kind} changes {changed:.2%} of the pixels")
            n = (shadowed(sides[1], index) if kind == "light" else
                 sum(shadowed(sides[1], li, by=index) for li in range(len(sides[1].lights))) if kind == "object" else None)
            assert n != 0, (rung, f"the added {kind} shadows no pixel")
            print(rung, f"added {kind} {index}: {changed:.1%} of the pixels change, {n} sampled pixels in its shadow")
        if rung == "spheres":   # the sphere at 1e30 is out of view and shadows nothing
            assert np.array_equal(images[1], images[2])
        if rung == "depth":
            side = sides[1]
            with pytest.raises(capi.RayHsError):
                rh.render(rh.Rendering(side.rs, side.rs.camera, W, H, 31))
    finally:
        for side in sides:
            side.rs.close()
