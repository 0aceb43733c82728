"""Built scenes with non-finite and extreme values in the places rh_scene_create accepts any double: material colours,
ior and checker size, texels, light colours, radii and positions, plane and mesh normals.  Shared by the value-domain
tests (tests/test_value_domain_gpu.py against the oracle, tests/test_value_domain_cpu.py for the oracle and the flatten).
The geometry is deliberately plain; only the values are at the edges.

Every case is (name, scene factory, max_depths, exact): `exact` when the scene has no reflective material, so that
every term of every sample has weight 1 at any max_depth (as at max_depth 0 in every scene) and finite linear colours
must equal the oracle's bit for bit."""
import math

import numpy as np

from tests.util import RawScene, grid_mesh

INF, NAN = math.inf, math.nan
W, H = 64, 48
BIG = 1e200  # BIG * BIG overflows, BIG alone does not

PLANE = {"kind": "plane", "point": (0, 0, 1.5), "normal": (0, 0, -1), "tangent": (1, 0, 0)}
FLOOR = {"kind": "plane", "point": (0, -0.7, 0), "normal": (0, 1, 0), "tangent": (1, 0, 0)}
SPHERE_C = (-0.5, 0.1, 0.6)
SPHERE = {"kind": "sphere", "center": SPHERE_C, "radius": 0.4}


def small_mesh(material, normals=None):
    g = grid_mesh(4, z=0.0, wobble=0.05, seed=7)
    g["positions"] = np.asarray(g["positions"]) * 0.35 + np.array([0.55, -0.1, 0.9])
    if normals is not None:
        g["normals"] = normals(np.asarray(g["normals"]))
    return dict(kind="mesh", material=material, **g)


def scene(objs, mats, lights, textures=(), camera=None):
    return RawScene(objs, mats, lights, textures=textures, camera=camera, size=(W, H, 0))


def with_mat(o, m):
    return dict(o, material=m)


# ---------------------------------------------------------------- finding 1: the Lambert cull of overflowing products
def lambert(sign, kind, cmap, n_lights=3):
    """A plane and a sphere lit from behind (a point light behind the plane, one at the sphere's centre, a directional
    light from behind the plane): their l.n <= 0 pairs are unoccluded, and cd (*) lc overflows in red."""
    cd = (sign * BIG, 0.5, 0.5)
    m = {"kind": kind, "cmap": cmap, "color1": cd, "color2": cd, "size": 0.4, "ior": 1.5}
    if cmap == "texture":
        m["texture"] = 0
    lc = (BIG, 1.0, 1.0)
    lights = [{"kind": "point", "vec": (0.2, 0.1, 3.0), "color": lc, "radius": 1.0},
              {"kind": "point", "vec": SPHERE_C, "color": lc, "radius": 1.0},
              {"kind": "directional", "vec": (0.1, 0.2, 1.0), "color": lc}]
    rng = np.random.RandomState(n_lights)
    while len(lights) < n_lights:   # ordinary lights in front, to reach the global-memory tables and the simple kernel
        lights.append({"kind": "point", "vec": tuple(rng.uniform(-1, 1, 3) * (1.5, 1, 0.5) + (0, 0, -1.5)),
                       "color": (0.05, 0.05, 0.05), "radius": 0.5})
    tex = [np.tile(np.array(cd), (2, 2, 1))] if cmap == "texture" else ()
    return scene([with_mat(PLANE, 0), with_mat(SPHERE, 0)], [m], lights, textures=tex)


# ---------------------------------------------------------------- finding 2: black under a non-finite factor
def specular(kind, ior):
    """One sphere of `kind` with `ior`, over a lit diffuse floor, with an emitter: reflection rays that miss, hit the
    floor or the emitter."""
    mats = [{"kind": kind, "ior": ior, "color1": (0.3, 0.6, 0.9)}, {"kind": "diffuse", "color1": (0.7, 0.7, 0.7)},
            {"kind": "emmit", "color1": (2.0, 1.5, 1.0)}]
    objs = [{"kind": "sphere", "center": (0, 0, 0.3), "radius": 0.6, "material": 0}, with_mat(FLOOR, 1),
            {"kind": "sphere", "center": (0.9, 0.5, -0.4), "radius": 0.2, "material": 2}]
    lights = [{"kind": "point", "vec": (0, 2, -1), "color": (3, 3, 3), "radius": 1.0}]
    return scene(objs, mats, lights)


# ---------------------------------------------------------------- light values
def lit_stage(light, extra_mats=()):
    """Diffuse plane, sphere and mesh, one ordinary light and the light under test."""
    mats = [{"kind": "diffuse", "color1": (0.8, 0.6, 0.4)}]
    objs = [with_mat(PLANE, 0), with_mat(SPHERE, 0), small_mesh(0)]
    lights = [{"kind": "point", "vec": (0.5, 1.0, -1.5), "color": (1.5, 1.5, 1.5), "radius": 1.0}, light]
    return scene(objs, mats, lights)


def centre_hit(rs):
    """The oracle's hit point of the middle pixel's camera ray."""
    from oracle.orc import OracleScene

    orc = OracleScene(rs.raw)
    o, d = orc.ray_from_pixel(rs.camera, W, H, W // 2, H // 2)
    return orc.closest(o, d)["p"]


def light_at_minus_distance():
    """A point light whose radius is exactly -dist(light, p) for the middle pixel's hit p: s = 0, falloff 1 / 0 = inf."""
    lp = (0.3, 0.4, -0.8)
    probe = lit_stage({"kind": "point", "vec": lp, "color": (1, 1, 1), "radius": 1.0})
    p = centre_hit(probe)
    dx, dy, dz = lp[0] - p[0], lp[1] - p[1], lp[2] - p[2]
    dd = math.sqrt(dx * dx + dy * dy + dz * dz)  # dist, Vec.hs:118-122, left to right
    return lit_stage({"kind": "point", "vec": lp, "color": (1, 1, 1), "radius": -dd})


def point(vec=(0.3, 0.4, -0.8), color=(1.0, 0.8, 0.6), radius=1.0):
    return {"kind": "point", "vec": vec, "color": color, "radius": radius}


def directional(vec, color=(0.7, 0.7, 0.7)):
    return {"kind": "directional", "vec": vec, "color": color}


LIGHTS = {
    "colour_inf": point(color=(INF, 1, 1)), "colour_-inf": point(color=(1, -INF, 1)), "colour_nan": point(color=(1, 1, NAN)),
    "dir_colour_inf": directional((0.2, 0.5, -1), color=(INF, -INF, 1)), "dir_colour_nan": directional((0.2, 0.5, -1), color=(NAN, 1, 1)),
    "radius_0": point(radius=0.0), "radius_-0": point(radius=-0.0), "radius_neg": point(radius=-0.5),
    "radius_inf": point(radius=INF), "radius_nan": point(radius=NAN), "radius_tiny": point(radius=1e-300),
    "at_1e200": point(vec=(0, BIG, 0)), "at_1e200_radius_inf": point(vec=(0, BIG, 0), radius=INF),
    "at_nan": point(vec=(NAN, 0.4, -0.8)),
    "dir_zero": directional((0.0, 0.0, 0.0)), "dir_subnormal": directional((5e-324, 1e-310, -5e-324)),
    "dir_small": directional((0.2e-3, 0.5e-3, -1e-3)), "dir_huge": directional((0.2 * BIG, 0.5 * BIG, -BIG)),
    "dir_inf": directional((0.2, INF, -1)), "dir_nan": directional((0.2, 0.5, NAN)),
}


# ---------------------------------------------------------------- material values
def colour_stage(mat, textures=()):
    """The material under test on the plane, the mesh and (flat colours only) the sphere, lit by two ordinary lights.
    The sphere's uv goes through atan / acos, whose libm differs between device and host (DESIGN §3), so a checker or
    texture there would test that instead of the values."""
    lights = [point(vec=(0.5, 1.0, -1.5), color=(1.5, 1.5, 1.5)), directional((-0.3, 0.6, -1), color=(0.4, 0.4, 0.4))]
    sphere = 0 if mat.get("cmap", "flat") == "flat" else 1
    return scene([with_mat(PLANE, 0), with_mat(SPHERE, sphere), small_mesh(0)], [mat, {"kind": "diffuse", "color1": (0.5, 0.5, 0.5)}],
                 lights, textures=textures)


def checker(size):
    return colour_stage({"kind": "diffuse", "cmap": "checker", "color1": (0.9, 0.2, 0.1), "color2": (0.1, 0.3, 0.9), "size": size})


def texture(texels):
    return colour_stage({"kind": "diffuse", "cmap": "texture", "texture": 0}, textures=[np.asarray(texels, dtype=np.float64)])


def flat(kind, color):
    return colour_stage({"kind": kind, "ior": 1.5, "color1": color})


MATERIALS = {  # name: (factory, args)
    "negative": (flat, ("diffuse", (-0.5, -2.0, -0.001))), "over_one": (flat, ("diffuse", (1.5, 7.0, 1.0000001))),
    "big": (flat, ("diffuse", (BIG, -BIG, 0.5))), "inf": (flat, ("diffuse", (INF, -INF, 0.5))),
    "nan": (flat, ("diffuse", (NAN, 0.5, 0.5))), "plastic_inf": (flat, ("plastic", (INF, 0.5, -INF))),
    "checker_0": (checker, (0.0,)), "checker_neg": (checker, (-0.3,)), "checker_tiny": (checker, (1e-300,)),
    "checker_huge": (checker, (1e300,)), "checker_inf": (checker, (INF,)), "checker_nan": (checker, (NAN,)),
    "texture_1x1": (texture, ([[[0.2, 0.7, -0.4]]],)),
    "texture_1xN": (texture, ([[[0.1, 0.2, 0.3], [0.9, -0.5, 0.1], [0.4, 0.4, 2.0]]],)),
    "texture_inf": (texture, ([[[INF, 0.2, 0.3], [0.5, 0.5, 0.5]], [[0.1, -INF, 0.2], [0.3, 0.3, 0.3]]],)),
    "texture_nan": (texture, ([[[NAN, 0.2, 0.3], [0.5, 0.5, 0.5]], [[0.1, 0.2, 0.2], [0.3, NAN, 0.3]]],)),
}


# ---------------------------------------------------------------- normals
def plane_normal(n):
    mats = [{"kind": "diffuse", "color1": (0.8, 0.6, 0.4)}, {"kind": "mirror", "ior": 2.0}]
    objs = [dict(PLANE, normal=n, material=0), with_mat(FLOOR, 1), with_mat(SPHERE, 0)]
    lights = [point(vec=(0.5, 1.0, -1.5), color=(1.5, 1.5, 1.5)), directional((-0.3, 0.6, -1), color=(0.4, 0.4, 0.4))]
    return scene(objs, mats, lights)


def mesh_normals(fill):
    """A Mirror mesh whose vertex normals are partly `fill` (zero, NaN or inf): NaN reflection rays."""
    def edit(nrm):
        nrm = nrm.copy()
        nrm[::3] = fill
        return nrm
    mats = [{"kind": "diffuse", "color1": (0.8, 0.6, 0.4)}, {"kind": "mirror", "ior": 2.0}, {"kind": "plastic", "ior": 1.4, "color1": (0.2, 0.5, 0.3)}]
    objs = [with_mat(PLANE, 0), with_mat(SPHERE, 0), small_mesh(1, edit), dict(small_mesh(2, edit), positions=np.asarray(small_mesh(2)["positions"]) - (1.0, 0.6, 0))]
    lights = [point(vec=(0.5, 1.0, -1.5), color=(1.5, 1.5, 1.5))]
    return scene(objs, mats, lights)


NORMALS = {
    "plane_small": (plane_normal, ((0, 0, -1e-3),)), "plane_large": (plane_normal, ((0, 0, -1e3),)),
    "plane_huge": (plane_normal, ((0, 0, -1e100),)), "plane_nan": (plane_normal, ((NAN, 0, -1),)),
    "mesh_zero": (mesh_normals, (0.0,)), "mesh_nan": (mesh_normals, (NAN,)), "mesh_inf": (mesh_normals, (INF,)),
}


# ---------------------------------------------------------------- toIntC
def show_uv():
    """An orthographic ShowUV plane whose u, v run over about [-2, 3] x [-1.4, 2.4]: hundreds of k/255 boundaries."""
    k = 5.0 / W
    objs = [{"kind": "plane", "point": (-0.5 / k, -0.5 / k, 1.0), "normal": (0, 0, -1), "tangent": (k, 0, 0), "material": 0}]
    return scene(objs, [{"kind": "showuv"}], [], camera={"position": (0, 0, -2), "projection": "orthographic"})


EMMIT_VALUES = [(1 / 255, 2 / 255, 128 / 255), (1.0, 254 / 255, 255 / 255), (math.nextafter(1.0, 2.0), 0.5, 0.25),
                (-1 / 255, -0.999 / 255, -0.0), (-INF, 0.0, 1.0), (100 / 255, 37 / 255, 200 / 255)]


def emitters():
    mats = [{"kind": "emmit", "color1": c} for c in EMMIT_VALUES]
    objs = [{"kind": "sphere", "center": (-1.25 + 0.5 * i, 0, 0.5), "radius": 0.24, "material": i} for i in range(len(mats))]
    return scene(objs, mats, [])


def cases():
    """(name, scene factory, max_depths, exact) of every value case."""
    out = []
    for sign in (1, -1):
        for kind in ("diffuse", "plastic"):
            for cmap in ("flat", "checker", "texture"):
                out.append((f"lambert_{kind}_{cmap}_{'+' if sign > 0 else '-'}", lambda s=sign, k=kind, c=cmap: lambert(s, k, c),
                            (0, 2) if kind == "plastic" else (0,), kind == "diffuse"))
        for n in (13, 40):
            out.append((f"lambert_{n}_lights_{'+' if sign > 0 else '-'}", lambda s=sign, n=n: lambert(s, "diffuse", "flat", n), (0,), True))
    for kind in ("mirror", "plastic", "transparent"):
        for ior in (1.0, 0.0, 0.5, -1.0, 1e300, INF, NAN):
            out.append((f"{kind}_ior_{ior}", lambda k=kind, i=ior: specular(k, i), (0, 1, 3), False))
    for name in LIGHTS:
        out.append((f"light_{name}", lambda n=name: lit_stage(LIGHTS[n]), (0,), True))
    out.append(("light_radius_minus_distance", light_at_minus_distance, (0,), True))
    for name, (f, args) in MATERIALS.items():
        out.append((f"material_{name}", lambda f=f, a=args: f(*a), (0, 2) if name == "plastic_inf" else (0,), name != "plastic_inf"))
    for name, (f, args) in NORMALS.items():
        # (NaN / inf mesh normals reflect into NaN rays, whose reference hits are the documented departure of DESIGN §3:
        # those cases stop at max_depth 0)
        depths = (0,) if name.startswith("mesh_") and name != "mesh_zero" else (0, 1, 3)
        out.append((f"normal_{name}", lambda f=f, a=args: f(*a), depths, False))
    # (the Lambert cases' texture is on the sphere too, but every texel there is the same colour)
    out.append(("toint_showuv", show_uv, (0,), True))
    out.append(("toint_emmit", emitters, (0,), True))
    return out
