"""Cost of sphere lights (RH_LIGHT_SPHERE) against the point lights they are made of.

    python scripts/sphere_light_rate.py [--pack tests/golden/dragon_full.pack] [--size 3840x2160] [--spp 16] [--json out.json]

Workload: dragon_full at 3840×2160, 16 spp, RH_OFFSETS_SPLITMIX64 with seed 24, device outputs.  Two configurations: the
pack's point lights, and the same lights as sphere lights of their own radius.  Sphere lights have no cube maps and no
lit-triangle flags, and their shadow rays diverge, so more (hit, light) pairs walk a tree; how much that costs is what
this measures.  Each configuration renders on its own copy of the scene.  After --warmup frames of each, --reps rounds
alternate the two; each frame is timed on the host clock around the call (it returns when the frame is complete), and
the best and all times are reported with Mrays/s (all classes over the best time), the rays per class, the shadow walk
pairs against the pairs the Lambert cull settled (rh_stats shadow_walk_pairs, rays_shadow_culled), the shadow schedule
and the queue factor.  One more frame of each with RH_FLAG_PROFILE (every launch timed on its own) gives the trace and
shadow kernels' times and the shadow kernels' share.  Parity: rows --rows of the last timed frame against the
sphere-light oracle's render of the same rows and seed (tests/sphere_light_oracle.py).  The card's name and power limit
are read in the same run.
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

import rayhs_b200 as rh  # noqa: E402
from rayhs_b200 import capi  # noqa: E402
from scripts.ray_query_rate import card  # noqa: E402
from tests.sphere_light_oracle import SphereOracle  # noqa: E402

CLASSES = ("rays_primary", "rays_reflect", "rays_probe", "rays_exit", "rays_shadow")


def scene(pack, spheres):
    sc = rh.Scene.from_pack(pack)
    if spheres:
        lights = sc.lights
        for L in lights:
            if L.kind == capi.RH_LIGHT_POINT:
                L.kind = capi.RH_LIGHT_SPHERE
        sc.update(lights=list(lights))
    return sc


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--pack", default=os.path.join(ROOT, "tests", "golden", "dragon_full.pack"))
    ap.add_argument("--size", default="3840x2160")
    ap.add_argument("--spp", type=int, default=16)
    ap.add_argument("--seed", type=int, default=24)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=4)
    ap.add_argument("--rows", type=int, nargs=3, default=[7, 2160, 1080], help="start, stop, step of the parity rows")
    ap.add_argument("--json", default=None, help="also write the result here")
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("sphere_light_rate.py measures on the GPU; no CUDA device here")
    w, h = (int(x) for x in a.size.split("x"))
    configs = {"point": scene(a.pack, False), "sphere": scene(a.pack, True)}
    res = {"card": card(), "pack": os.path.basename(a.pack), "width": w, "height": h, "spp": a.spp, "seed": a.seed, "configs": {}}
    jobs = {tag: rh.renderingFromScene(sc, w, h) for tag, sc in configs.items()}
    rgb = {tag: torch.empty((h, w, 3), dtype=torch.uint8, device="cuda") for tag in configs}
    for tag in configs:
        for _ in range(a.warmup):
            rh.render_device(jobs[tag], rgb[tag], spp=a.spp, seed=a.seed)
    times = {tag: [] for tag in configs}
    stats = {}
    for _ in range(a.reps):
        for tag in configs:
            t0 = time.perf_counter()
            stats[tag] = rh.render_device(jobs[tag], rgb[tag], spp=a.spp, seed=a.seed)
            times[tag].append((time.perf_counter() - t0) * 1e3)
    for tag, sc in configs.items():
        st = stats[tag]
        prof_rgb = torch.empty_like(rgb[tag])
        prof = rh.render_device(jobs[tag], prof_rgb, spp=a.spp, seed=a.seed, profile=True)
        rays = {k: int(st[k]) for k in CLASSES}
        best = min(times[tag])
        ref = SphereOracle(sc.raw).render_sample(sc.camera, w, h, sc.max_depth, a.spp, a.seed, rows=tuple(a.rows))
        got = rgb[tag].cpu().numpy()[ref["rows"]]
        d = np.abs(got.astype(np.int32) - ref["rgb_u8"].astype(np.int32))
        ms_trace, ms_shadow = float(prof["ms_trace"]), float(prof["ms_shadow"])
        run = {"ms_best": best, "ms_all": times[tag], "ms_total": st["ms_total"], "mrays_per_s": sum(rays.values()) / best / 1e3,
               "rays": rays, "shadow_walk_pairs": int(st["shadow_walk_pairs"]), "shadow_culled_pairs": int(st["rays_shadow_culled"]),
               "shadow_split": int(st["shadow_split"]), "queue_factor": st["queue_factor"],
               "profile_ms_trace": ms_trace, "profile_ms_shadow": ms_shadow, "profile_shadow_share": ms_shadow / (ms_trace + ms_shadow),
               "profile_same_bytes": bool(torch.equal(prof_rgb, rgb[tag])),
               "parity_rows": [int(r) for r in ref["rows"]], "parity_exact": float((d == 0).mean()), "parity_max_diff": int(d.max())}
        res["configs"][tag] = run
        print(f"{tag:7s}: {best:8.2f} ms ({run['mrays_per_s']:8.1f} Mrays/s), walk pairs {run['shadow_walk_pairs']}, culled "
              f"{run['shadow_culled_pairs']}, shadow share {run['profile_shadow_share']:.3f}, parity exact {run['parity_exact']:.6f} "
              f"max diff {run['parity_max_diff']}", file=sys.stderr)
    res["cost_sphere_vs_point"] = res["configs"]["sphere"]["ms_best"] / res["configs"]["point"]["ms_best"]
    line = json.dumps(res)
    print(line)
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
