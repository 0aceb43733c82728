"""Shared helpers of the parity tests: scene packs, the oracle, and the comparison metrics of
BASELINE.json (hit ids bit-exact; <= 1 LSB on >= 99.9 % of pixels; PSNR >= 50 dB)."""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SCENES = ["cornellBox", "texture", "transform", "dragon_superlow", "dragon_low", "dragon_full", "outScene"]


def load_scene(name):
    from rayhs_b200 import Scene

    return Scene.from_pack(os.path.join(GOLDEN, name + ".pack"))


def temp_library(name, sources, flags):
    """Compiles sources[0] (which includes the rest of `sources`) with the C++ compiler into a shared library in the
    temporary directory, named by a digest of the sources and flags, so that the repository tree is never written, and
    loads it.  The rename makes the build safe against concurrent test processes."""
    h = hashlib.sha256(" ".join(flags).encode())
    for s in sources:
        with open(s, "rb") as f:
            h.update(f.read())
    path = os.path.join(tempfile.gettempdir(), f"rayhs_{name}_{os.getuid()}_{h.hexdigest()[:16]}.so")
    if not os.path.exists(path):
        tmp = f"{path}.{os.getpid()}"
        subprocess.check_call([os.environ.get("CXX") or "g++", *flags, sources[0], "-o", tmp, "-lpthread"])
        os.replace(tmp, path)
    return ctypes.CDLL(path)


def oracle_for(scene):
    from oracle.orc import OracleScene

    return OracleScene(scene.raw)


def psnr(a, b):
    mse = np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2)
    return float("inf") if mse == 0 else 10 * np.log10(255.0 ** 2 / mse)


def compare_images(gpu_u8, ref_u8):
    diff = np.abs(gpu_u8.astype(np.int32) - ref_u8.astype(np.int32)).max(axis=-1)
    return dict(exact=float(np.mean(diff == 0)), within1=float(np.mean(diff <= 1)), maxdiff=int(diff.max()),
                psnr=psnr(gpu_u8, ref_u8))


def assert_parity(gpu_u8, ref_u8, what=""):
    m = compare_images(gpu_u8, ref_u8)
    assert m["within1"] >= 0.999, (what, m)   # BASELINE.json: <= 1 LSB per channel on >= 99.9 % of pixels
    assert m["psnr"] >= 50.0, (what, m)       # BASELINE.json: PSNR >= 50 dB
    return m


# The tolerance of a linear colour against the oracle's (tests/test_pyref_pins_oracle.py uses it too): the wavefront adds
# a sample's terms in its own order, <= 1 ulp per term, and Transparent forks with atomics (DESIGN §3).
RTOL, ATOL = 1e-9, 1e-12


def to_int_c(c):
    """Image.hs:54-55 toIntC, clamped into 0..255 as rh_render stores it (NaN: hs_min NaN 1 = 1, so 255)."""
    v = 255 * np.where(c <= 1, c, 1.0)
    return np.where(v < 0, 0, np.minimum(np.trunc(np.where(v < 0, 0, v)), 255)).astype(np.uint8)


def assert_oracle_exact(pixels, linear, ref, what=""):
    """The image equals the oracle's (`ref`: OracleScene.render) up to the departures of DESIGN §3, channel by channel:
    the linear colour is within RTOL / ATOL of the oracle's (NaN equals NaN); the bytes are toIntC of the device's own
    linear colour; and they are the oracle's bytes, except where the two linear colours, that close, straddle a
    quantisation step — there they differ by exactly 1.  Returns the number of such straddled channels."""
    want_lin, want_u8 = ref["rgb_f64"], ref["rgb_u8"]
    linear = np.asarray(linear, dtype=np.float64).reshape(want_lin.shape)
    pixels = np.asarray(pixels).reshape(want_u8.shape)
    ok = np.isclose(linear, want_lin, rtol=RTOL, atol=ATOL, equal_nan=True)
    bad = np.argwhere(~ok)[:5]
    assert ok.all(), (what, f"{int((~ok).sum())} linear channels off the oracle's", bad.tolist(),
                      [(linear[tuple(b)], want_lin[tuple(b)]) for b in bad])
    own = to_int_c(linear)
    bad = np.argwhere(pixels != own)[:5]
    assert not len(bad), (what, f"{int((pixels != own).sum())} bytes are not toIntC of the linear colour", bad.tolist(),
                          [(int(pixels[tuple(b)]), int(own[tuple(b)]), linear[tuple(b)]) for b in bad])
    straddled = own != to_int_c(want_lin)
    d = pixels.astype(np.int32) - want_u8.astype(np.int32)
    wrong = np.where(straddled, np.abs(d) != 1, d != 0)
    bad = np.argwhere(wrong)[:5]
    assert not wrong.any(), (what, f"{int(wrong.sum())} bytes off the oracle's ({int(straddled.sum())} channels straddle a "
                                   "quantisation step and may differ by 1)", bad.tolist(),
                             [(int(pixels[tuple(b)]), int(want_u8[tuple(b)])) for b in bad])
    return int(straddled.sum())


def render_linear(job, spp=1, offsets=None, seed=None, **kw):
    """The frame rh_render makes (progressive rendering's first call traces the same samples and stores the same bytes;
    tests/test_accumulate_gpu.py pins that) with its linear colours, hit ids and stats.  `seed`: the samples of
    sample_offsets(width * height, spp, seed), regenerated on the device."""
    import rayhs_b200 as rh

    acc = rh.Accumulator(job, stream_spp=spp if seed is not None else 0)
    try:
        return acc.add(spp, offsets=offsets, seed=seed, want_hit_ids=True, **kw)
    finally:
        acc.close()


# ---------------------------------------------------------------------------------------------
# Hand-built raw scenes (rh_raw_scene) for analytic and edge-case tests.
class RawScene:
    """Keeps the ctypes arrays of an rh_raw_scene alive.  objects: list of dicts
    {kind:'plane'|'sphere'|'mesh', material:int, a,b,c (plane: point, normal, tangent; sphere: center, radius),
     positions [n,3], normals [n,3], uvs [n,2], indices [m]}; materials: list of dicts; lights: list of dicts."""

    def __init__(self, objects, materials, lights, textures=(), camera=None, size=(64, 64, 3)):
        import ctypes as C

        from rayhs_b200 import capi

        self._keep = []
        n = len(objects)
        objs = (capi.rh_raw_object * max(n, 1))()
        for i, o in enumerate(objects):
            ro = objs[i]
            ro.kind = {"plane": capi.RH_OBJ_PLANE, "sphere": capi.RH_OBJ_SPHERE, "mesh": capi.RH_OBJ_MESH}[o["kind"]]
            ro.material = o.get("material", 0)
            if o["kind"] == "plane":
                ro.a[:], ro.b[:], ro.c[:] = o["point"], o["normal"], o["tangent"]
            elif o["kind"] == "sphere":
                ro.a[:] = o["center"]
                ro.b[:] = (o["radius"], 0.0, 0.0)
            else:
                pos = np.ascontiguousarray(o["positions"], dtype=np.float64).reshape(-1, 3)
                nrm = np.ascontiguousarray(o.get("normals", np.zeros_like(pos)), dtype=np.float64).reshape(-1, 3)
                uv = np.ascontiguousarray(o.get("uvs", np.zeros((len(pos), 2))), dtype=np.float64).reshape(-1, 2)
                idx = np.ascontiguousarray(o["indices"], dtype=np.uint32).reshape(-1)
                self._keep += [pos, nrm, uv, idx]
                ro.n_verts, ro.n_indices = len(pos), len(idx)
                ro.positions = pos.ctypes.data_as(C.POINTER(C.c_double))
                ro.normals = nrm.ctypes.data_as(C.POINTER(C.c_double))
                ro.uvs = uv.ctypes.data_as(C.POINTER(C.c_double))
                ro.indices = idx.ctypes.data_as(C.POINTER(C.c_uint32))
        mats = (capi.rh_material * max(len(materials), 1))()
        kinds = {"mirror": 0, "diffuse": 1, "plastic": 2, "emmit": 3, "transparent": 4, "shownormal": 5, "showuv": 6}
        cmaps = {"flat": 0, "checker": 1, "texture": 2}
        for i, m in enumerate(materials):
            mm = mats[i]
            mm.kind = kinds[m["kind"]]
            mm.cmap_kind = cmaps[m.get("cmap", "flat")]
            mm.ior = m.get("ior", 1.5)
            mm.color1[:] = m.get("color1", (1, 1, 1))
            mm.color2[:] = m.get("color2", (0, 0, 0))
            mm.size = m.get("size", 1.0)
            mm.texture = m.get("texture", -1)
        lts = (capi.rh_light * max(len(lights), 1))()
        for i, l in enumerate(lights):
            ll = lts[i]
            ll.kind = capi.RH_LIGHT_POINT if l["kind"] == "point" else capi.RH_LIGHT_DIRECTIONAL
            ll.vec[:] = l["vec"]
            ll.color[:] = l.get("color", (1, 1, 1))
            ll.radius = l.get("radius", 1.0)
        texs = (capi.rh_texture * max(len(textures), 1))()
        texels = []
        for i, t in enumerate(textures):
            arr = np.asarray(t, dtype=np.float64)  # [h, w, 3]
            texs[i].h, texs[i].w, texs[i].offset = arr.shape[0], arr.shape[1], sum(len(x) for x in texels) // 3
            texels.append(arr.reshape(-1))
        tex_arr = np.ascontiguousarray(np.concatenate(texels) if texels else np.zeros(3))
        self._keep += [objs, mats, lts, texs, tex_arr]
        raw = capi.rh_raw_scene()
        raw.n_objects, raw.n_materials, raw.n_lights, raw.n_textures = n, len(materials), len(lights), len(textures)
        raw.objects, raw.materials, raw.lights, raw.textures = objs, mats, lts, texs
        raw.texels = tex_arr.ctypes.data_as(C.POINTER(C.c_double))
        raw.n_texels = (len(tex_arr) // 3) if texels else 0
        self.raw_struct = raw
        self.raw = C.pointer(raw)
        cam = capi.rh_camera()
        c = camera or {}
        cam.position[:] = c.get("position", (0, 0, -2))
        cam.target[:] = c.get("target", (0, 0, 0))
        cam.up[:] = c.get("up", (0, 1, 0))
        cam.projection = capi.RH_PROJ_ORTHOGRAPHIC if c.get("projection") == "orthographic" else capi.RH_PROJ_PERSPECTIVE
        cam.fovy = c.get("fovy", 0.9272952180016123)
        self.camera = cam
        self.width, self.height, self.max_depth = size
        self._flat = None
        self._dev = None

    # the same views rayhs_b200.Scene offers, so that rh.render() can take a RawScene
    @property
    def flat(self):
        import ctypes as C

        from rayhs_b200 import capi

        if self._flat is None:
            self._flat = C.c_void_p()
            capi.check(capi.lib().rh_flatten(self.raw, C.byref(self._flat)))
        return capi.lib().rh_flat_desc(self._flat)

    @property
    def device(self):
        import ctypes as C

        import rayhs_b200 as rh
        from rayhs_b200 import capi

        if self._dev is None:
            rh.init()
            self._dev = C.c_void_p()
            capi.check(capi.lib().rh_scene_create(self.flat, C.byref(self._dev)))
        return self._dev

    def close(self):
        """Releases the device scene and the flattened scene (a scene with many light maps holds hundreds of MB)."""
        from rayhs_b200 import capi

        if self._dev:
            capi.lib().rh_scene_destroy(self._dev)
        if self._flat:
            capi.lib().rh_flat_destroy(self._flat)
        self._dev = self._flat = None


def grid_mesh(n, z=0.0, wobble=0.0, seed=1):
    """n x n quads (2 n^2 triangles) on [-1,1]^2: enough triangles for a real tree (>= 20 per split)."""
    rng = np.random.RandomState(seed)
    xs = np.linspace(-1, 1, n + 1)
    pos = np.array([(x, y, z + wobble * rng.uniform(-1, 1)) for y in xs for x in xs])
    nrm = np.tile((0.0, 0.0, -1.0), (len(pos), 1)) + 0.2 * rng.uniform(-1, 1, size=(len(pos), 3))
    uv = (pos[:, :2] + 1) / 2
    idx = []
    for j in range(n):
        for i in range(n):
            a = j * (n + 1) + i
            idx += [a, a + 1, a + n + 2, a, a + n + 2, a + n + 1]
    return dict(positions=pos, normals=nrm, uvs=uv, indices=idx)
