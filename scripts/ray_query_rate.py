"""Rates of the batched ray queries (rh_closest_intersection / rh_shadow_intersection) on the bench scene, beside the
closest-hit rate of a rendered frame of the same view.

    python scripts/ray_query_rate.py [--pack tests/golden/dragon_full.pack] [--width 3840 --height 2160] [--json out.json]

Workloads:
  (a) camera rays of the bench view through the pixel coordinates rayTrace uses (Image.hs:31-36): coherent;
  (b) incoherent rays: origins uniform in the scene's bounds, uniform unit directions (seeded);
  (c) shadow queries towards each light from the hits of (a) (accumDiffuse's rayEps p ld, RayHs.hs:89-97).
For each: Mrays/s with device buffers (CUDA events around the call, after a warm-up call) and with host buffers (numpy
in and out, host clock around the call, which returns when the results are written).  Comparison: a profiled 1-spp
rh_render of the same view, its closest-hit rays (primary + reflect + probe + exit) over its ms_trace (closest-hit +
shade kernels).  The card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import rayhs_b200 as rh  # noqa: E402


def camera_rays(cam, w: int, h: int) -> np.ndarray:
    """rayFromPixel (Projection.hs:22-46, Mat.hs:83-93) for every pixel (x, y), row-major: [w*h, 6]."""
    pos, target, up = (np.array(v[:], dtype=np.float64) for v in (cam.position, cam.target, cam.up))
    aspect = w / h
    apw, aph = (w, w / aspect) if aspect > 1 else (aspect * h, h)
    py, px = np.mgrid[0:h, 0:w].astype(np.float64)
    x, y = apw * (px.ravel() - w / 2) / w, aph * (-py.ravel() + h / 2) / h
    n = w * h
    if cam.projection == rh.capi.RH_PROJ_ORTHOGRAPHIC:
        o = np.stack([x, y, np.zeros(n)], axis=1)
        d = np.tile([0.0, 0.0, 1.0], (n, 1))
    else:
        f = 0.5 * h / (math.tan(0.5) * cam.fovy)
        v = np.stack([x, y, np.full(n, f)], axis=1)
        d = v / np.sqrt((v * v).sum(axis=1))[:, None]
        o = np.zeros((n, 3))

    def normalize(a):
        return a / math.sqrt(float(a @ a))

    forward = normalize(target - pos)
    right = normalize(np.cross(up, forward))
    upv = np.cross(forward, right)
    m = np.stack([right, upv, forward], axis=1)  # fromColumns right up forward
    return np.concatenate([o + pos, d @ m.T], axis=1)


def shadow_rays(p: np.ndarray, light) -> np.ndarray:
    """rayEps p ld towards one light (Light.hs:12-17)."""
    v = np.array(light.vec[:], dtype=np.float64)
    if light.kind == rh.capi.RH_LIGHT_DIRECTIONAL:
        ld = np.broadcast_to(v, p.shape)
    else:
        w = v - p
        ld = w / np.sqrt((w * w).sum(axis=1))[:, None]
    return np.concatenate([p + 1e-6 * ld, ld], axis=1)


def card() -> dict:
    import torch

    out = {"name": torch.cuda.get_device_name(), "power_limit_w": None}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        out["power_limit_w"] = float(q.stdout.strip().splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        pass
    return out


def rate(sc, rays: np.ndarray, light: int | None, reps: int) -> dict:
    """Mrays/s of one query kind over `rays`, device buffers then host buffers (the best of `reps` timed calls each)."""
    import torch

    o, d = np.ascontiguousarray(rays[:, :3]), np.ascontiguousarray(rays[:, 3:])
    od, dd = torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda()

    def call(a, b):
        return rh.closestIntersection(sc, a, b) if light is None else rh.shadowIntersection(sc, light, a, b)

    call(od, dd)  # warm-up: module load, scratch allocation
    dev = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        call(od, dd)
        e1.record()
        e1.synchronize()
        dev.append(e0.elapsed_time(e1))
    call(o, d)
    host = []
    for _ in range(reps):
        t0 = time.perf_counter()
        call(o, d)
        host.append((time.perf_counter() - t0) * 1e3)
    n = len(rays)
    return {"rays": n, "ms_device": min(dev), "ms_host": min(host), "mrays_s_device": n / min(dev) / 1e3,
            "mrays_s_host": n / min(host) / 1e3, "ms_device_all": dev, "ms_host_all": host}


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--pack", default=os.path.join(ROOT, "tests", "golden", "dragon_full.pack"))
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--incoherent", type=int, default=16 << 20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--seed", type=int, default=7)
    ap.add_argument("--json", default=None, help="also write the result here")
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("ray_query_rate.py measures on the GPU; no CUDA device here")
    sc = rh.Scene.from_pack(a.pack)
    flat = sc.flat.contents
    res = {"card": card(), "pack": os.path.basename(a.pack), "width": a.width, "height": a.height}

    # the render of the same view: 1 spp, every launch timed
    job = rh.renderingFromScene(sc, a.width, a.height)
    rh.render(job, profile=True)
    st = rh.render(job, profile=True).stats
    closest_rays = st["rays_primary"] + st["rays_reflect"] + st["rays_probe"] + st["rays_exit"]
    res["render_1spp"] = {"ms_trace": st["ms_trace"], "closest_hit_rays": closest_rays,
                          "mrays_s_trace": closest_rays / st["ms_trace"] / 1e3, "ms_total": st["ms_total"]}

    cam = camera_rays(sc.camera, a.width, a.height)
    res["a_camera"] = rate(sc, cam, None, a.reps)
    rng = np.random.default_rng(a.seed)
    pts = []
    raw = sc.raw.contents
    for i in range(raw.n_objects):
        ob = raw.objects[i]
        if ob.kind == rh.capi.RH_OBJ_MESH and ob.n_verts:
            pts.append(np.ctypeslib.as_array(ob.positions, shape=(ob.n_verts, 3)))
    pts = np.concatenate(pts)
    lo, hi = pts.min(axis=0), pts.max(axis=0)
    u = rng.normal(size=(a.incoherent, 3))
    inc = np.concatenate([rng.uniform(lo, hi, (a.incoherent, 3)), u / np.linalg.norm(u, axis=1, keepdims=True)], axis=1)
    del u
    res["b_incoherent"] = rate(sc, inc, None, a.reps)
    del inc
    hits = rh.closestIntersection(sc, cam[:, :3].copy(), cam[:, 3:].copy())
    p = hits.p[hits.object >= 0]
    res["c_shadow"] = []
    for li in range(flat.n_lights):
        r = rate(sc, shadow_rays(p, flat.lights[li]), li, a.reps)
        r["light"], r["kind"] = li, "point" if flat.lights[li].kind == rh.capi.RH_LIGHT_POINT else "directional"
        res["c_shadow"].append(r)
    res["camera_per_ray_vs_render"] = res["render_1spp"]["mrays_s_trace"] / res["a_camera"]["mrays_s_device"]
    line = json.dumps(res)
    print(line)
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
