"""Rates of the radiance queries (rh_trace_rays) on the bench scene, beside rh_render of the same view.

    python scripts/trace_rays_rate.py [--pack tests/golden/dragon_full.pack] [--width 3840 --height 2160] [--json out.json]

Workloads, all at the scene's own depth limit:
  (a) the camera rays of the bench view (scripts/ray_query_rate.py's camera_rays) through rh_trace_rays with device
      buffers, beside rh_render of the same view at 1 spp (RH_OFFSETS_NONE, device output): the same wavefront work;
  (b) incoherent rays, device buffers: origins uniform in the scene's bounds, uniform unit directions (seeded);
  (c) (a) and (b) with host buffers (numpy in and out; the rays stream in through the upload ring).
Device times are CUDA events around the call, host times a host clock around it (the call returns when the colours are
written); each is the best of --reps calls after warm-up calls, the render and the trace calls alternating.  The scene's
renders are warmed up first, so that its shadow-walk schedule is decided and both sides use the same one.  The card's
name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import rayhs_b200 as rh  # noqa: E402
from ray_query_rate import camera_rays, card  # noqa: E402

COUNTS = ("rays_primary", "rays_reflect", "rays_probe", "rays_exit", "rays_shadow", "rays_shadow_culled")


def timed(fn, device: bool) -> tuple[float, dict]:
    import torch

    if device:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        st = fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1), st
    t0 = time.perf_counter()
    st = fn()
    return (time.perf_counter() - t0) * 1e3, st


def summary(ms: list[float], st: dict, n: int) -> dict:
    best = min(ms)
    return {"rays": n, "ms": best, "mrays_s": n / best / 1e3, "ms_all": ms, "ms_total_stats": st["ms_total"],
            "chunks": st["chunks"], "queue_factor": st["queue_factor"], "shadow_split": st["shadow_split"],
            **{k: st[k] for k in COUNTS}}


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
        sys.exit("trace_rays_rate.py measures on the GPU; no CUDA device here")
    sc = rh.Scene.from_pack(a.pack)
    depth = sc.max_depth
    res = {"card": card(), "pack": os.path.basename(a.pack), "width": a.width, "height": a.height, "max_depth": depth}

    job = rh.renderingFromScene(sc, a.width, a.height)
    rgb = torch.empty((a.height, a.width, 3), dtype=torch.uint8, device="cuda")
    for _ in range(4):  # the scene's timing frames: afterwards its shadow-walk schedule is decided
        rh.render_device(job, rgb)

    cam = camera_rays(sc.camera, a.width, a.height)
    o, d = np.ascontiguousarray(cam[:, :3]), np.ascontiguousarray(cam[:, 3:])
    od, dd = torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda()

    def render():
        return rh.render_device(job, rgb)

    def trace_dev():
        return rh.traceRay(sc, od, dd, depth).stats

    def trace_host():
        return rh.traceRay(sc, o, d, depth).stats

    for f in (render, trace_dev, trace_host):
        f()
    ms = {"render": [], "trace_dev": [], "trace_host": []}
    last = {}
    for _ in range(a.reps):
        for name, f, dev in (("render", render, True), ("trace_dev", trace_dev, True), ("trace_host", trace_host, False)):
            t, last[name] = timed(f, dev)
            ms[name].append(t)
    n = len(cam)
    res["render_1spp"] = summary(ms["render"], last["render"], n)
    res["a_camera_device"] = summary(ms["trace_dev"], last["trace_dev"], n)
    res["c_camera_host"] = summary(ms["trace_host"], last["trace_host"], n)
    res["a_trace_over_render"] = res["a_camera_device"]["ms"] / res["render_1spp"]["ms"]
    del od, dd, o, d, cam

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
    o = rng.uniform(lo, hi, (a.incoherent, 3))
    d = u / np.linalg.norm(u, axis=1, keepdims=True)
    del u
    od, dd = torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda()
    ms = {"dev": [], "host": []}
    for _ in range(2):
        rh.traceRay(sc, od, dd, depth)
    rh.traceRay(sc, o, d, depth)
    for _ in range(a.reps):
        t, last["dev"] = timed(lambda: rh.traceRay(sc, od, dd, depth).stats, True)
        ms["dev"].append(t)
        t, last["host"] = timed(lambda: rh.traceRay(sc, o, d, depth).stats, False)
        ms["host"].append(t)
    res["b_incoherent_device"] = summary(ms["dev"], last["dev"], a.incoherent)
    res["c_incoherent_host"] = summary(ms["host"], last["host"], a.incoherent)
    line = json.dumps(res)
    print(line)
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
