"""Cost of thin-lens cameras (RH_PROJ_THIN_LENS) against the pinhole camera they are built on.

    python scripts/lens_rate.py [--pack tests/golden/dragon_full.pack] [--size 3840x2160] [--spp 16] [--json out.json]

Workload: dragon_full at 3840×2160, 16 spp, RH_OFFSETS_SPLITMIX64 with seed 24, device outputs.  Three cameras: the
pack's perspective camera, and thin lenses on it with the focus on the dragon (the distance along the view axis to the
first hit of the centre pixel's ray) at a small and a large aperture (--apertures, as fractions of that distance).
Lens primary rays are less coherent than pinhole ones, so their frames are expected to cost more; how much is what this
measures.  Each camera renders on its own copy of the scene, so that each learns its own shadow schedule and queue
factor.  After --warmup frames of each (module load, scratch, and the scene's shadow-schedule timing frames), --reps
rounds alternate the three cameras; each frame is timed on the host clock around the call (it returns when the frame is
complete), and the best and all times are reported with the frame's ms_total, the rays per class, Mrays/s (all classes
over the best time), the shadow schedule and the queue factor.  Parity: rows --rows of the last frame against the
oracle's render of the same rows and seed (tests/lens_oracle.py render_sample: the oracle with the lens ray) (bytes: exact share and largest difference).  The card's name and
power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import rayhs_b200 as rh  # noqa: E402
from oracle.orc import OracleScene, camera_rays  # noqa: E402
from tests import lens_oracle  # noqa: E402
from scripts.ray_query_rate import card  # noqa: E402

CLASSES = ("rays_primary", "rays_reflect", "rays_probe", "rays_exit", "rays_shadow")


def focus_on_the_centre(sc, w, h) -> tuple[float, int]:
    """(distance along the view axis to the first hit of the centre pixel's ray, object hit; -1 and the distance to the
    target on a miss)."""
    c = sc.camera
    ray = camera_rays(c, w, h, np.array([[w / 2, h / 2]]))
    hit = rh.closestIntersection(sc, np.ascontiguousarray(ray[:, :3]), np.ascontiguousarray(ray[:, 3:]))
    fwd = np.subtract(c.target, c.position)
    fwd = fwd / np.linalg.norm(fwd)
    if hit.object[0] < 0:
        return math.dist(c.position, c.target), -1
    return float(hit.t[0] * np.dot(ray[0, 3:], fwd)), int(hit.object[0])


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--pack", default=os.path.join(ROOT, "tests", "golden", "dragon_full.pack"))
    ap.add_argument("--size", default="3840x2160")
    ap.add_argument("--spp", type=int, default=16)
    ap.add_argument("--seed", type=int, default=24)
    ap.add_argument("--apertures", type=float, nargs=2, default=[0.005, 0.05])
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--rows", type=int, nargs=3, default=[7, 2160, 540], help="start, stop, step of the parity rows")
    ap.add_argument("--json", default=None, help="also write the result here")
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("lens_rate.py measures on the GPU; no CUDA device here")
    w, h = (int(x) for x in a.size.split("x"))
    probe = rh.Scene.from_pack(a.pack)
    focus, obj = focus_on_the_centre(probe, w, h)
    cams = {"perspective": probe.camera}
    for tag, frac in zip(("lens_small", "lens_large"), a.apertures):
        cams[tag] = rh.thinLens(probe.camera, frac * focus, focus)
    res = {"card": card(), "pack": os.path.basename(a.pack), "width": w, "height": h, "spp": a.spp, "seed": a.seed,
           "focus_distance": focus, "focus_object": obj, "cameras": {}}
    scenes = {tag: rh.Scene.from_pack(a.pack) for tag in cams}
    jobs = {tag: rh.Rendering(scenes[tag], cam, w, h, probe.max_depth) for tag, cam in cams.items()}
    rgb = {tag: torch.empty((h, w, 3), dtype=torch.uint8, device="cuda") for tag in cams}
    for tag in cams:
        for _ in range(a.warmup):
            rh.render_device(jobs[tag], rgb[tag], spp=a.spp, seed=a.seed)
    times = {tag: [] for tag in cams}
    stats = {}
    for _ in range(a.reps):
        for tag in cams:
            t0 = time.perf_counter()
            stats[tag] = rh.render_device(jobs[tag], rgb[tag], spp=a.spp, seed=a.seed)
            times[tag].append((time.perf_counter() - t0) * 1e3)
    rows = tuple(a.rows)
    orc = OracleScene(probe.raw)
    for tag, cam in cams.items():
        st = stats[tag]
        rays = {k: int(st[k]) for k in CLASSES}
        best = min(times[tag])
        ref = lens_oracle.render_sample(orc, cam, w, h, probe.max_depth, a.spp, a.seed, rows=rows)
        got = rgb[tag].cpu().numpy()[ref["rows"]]
        d = np.abs(got.astype(np.int32) - ref["rgb_u8"].astype(np.int32))
        run = {"projection": int(cam.projection), "aperture": cam.proj_width if cam.projection == rh.capi.RH_PROJ_THIN_LENS else 0.0,
               "ms_best": best, "ms_all": times[tag], "ms_total": st["ms_total"], "mrays_per_s": sum(rays.values()) / best / 1e3,
               "rays": rays, "shadow_split": int(st["shadow_split"]), "queue_factor": st["queue_factor"], "chunks": int(st["chunks"]),
               "parity_rows": [int(r) for r in ref["rows"]], "parity_exact": float((d == 0).mean()), "parity_max_diff": int(d.max())}
        res["cameras"][tag] = run
        print(f"{tag:12s} R={run['aperture']:.5f}: {best:8.2f} ms ({run['mrays_per_s']:8.1f} Mrays/s), shadow_split "
              f"{run['shadow_split']}, queue_factor {run['queue_factor']:.3f}, parity exact {run['parity_exact']:.6f} max diff "
              f"{run['parity_max_diff']}", file=sys.stderr)
    base = res["cameras"]["perspective"]["ms_best"]
    for run in res["cameras"].values():
        run["cost_vs_perspective"] = run["ms_best"] / base
    line = json.dumps(res)
    print(line)
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
