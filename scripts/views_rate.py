"""Cost of camera batches (rh_render_views) against one rh_render call per view.

    python scripts/views_rate.py [--pack tests/golden/dragon_full.pack] [--views 6 64 256] [--spp 1 16] [--json out.json]

Workload: the bench scene, V views around its camera (position and target moved by up to 0.3, as a rig or turntable
would), sizes 128², 256², 512² and 1920×1080, 1 and 16 spp, RH_OFFSETS_SPLITMIX64 with seed 24 + v for view v, device
outputs.  Each case loads the scene afresh, so that its renders use the queue factor their own frame size needs
rather than one a smaller case's renders left on the scene.  Per case, after a warm-up round of both (module load, scratch, and the renders' shadow-schedule timing
frames), --reps rounds alternate one renderViews call and V render_device calls into the slices of one [V, H, W, 3]
tensor; each is timed on the host clock around the calls (each call returns after its frame is complete) and the best
round is reported, with the batch's ms_total and the sum of the renders' ms_total beside it.  The outputs of the last
round are checked equal (and the largest byte difference recorded).  A case the device memory cannot hold at the time
(another process on the card) is recorded as such with the free memory, and the run goes on.  The card's name and power
limit are read in the same run.
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

SIZES = [(128, 128), (256, 256), (512, 512), (1920, 1080)]


def cameras(sc, V):
    rng = np.random.RandomState(V)
    out = []
    for v in range(V):
        c = capi.rh_camera.from_buffer_copy(sc.camera)
        d = rng.uniform(-0.3, 0.3, 3) if v else np.zeros(3)
        for k in range(3):
            c.position[k] += d[k]
            c.target[k] += 0.5 * d[k]
        out.append(c)
    return out


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--pack", default=os.path.join(ROOT, "tests", "golden", "dragon_full.pack"))
    ap.add_argument("--views", type=int, nargs="+", default=[6, 64, 256])
    ap.add_argument("--spp", type=int, nargs="+", default=[1, 16])
    ap.add_argument("--sizes", nargs="+", default=[f"{w}x{h}" for w, h in SIZES])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--json", default=None, help="also write the result here")
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("views_rate.py measures on the GPU; no CUDA device here")
    res = {"card": card(), "pack": os.path.basename(a.pack), "free_gb_at_start": torch.cuda.mem_get_info()[0] / 1e9, "runs": []}
    for size in a.sizes:
        w, h = (int(x) for x in size.split("x"))
        for spp in a.spp:
            for V in a.views:
                sc = rh.Scene.from_pack(a.pack)
                base = rh.renderingFromScene(sc, w, h)
                cams = cameras(sc, V)
                seeds = [24 + v for v in range(V)]
                jobs = [rh.Rendering(sc, c, w, h, base.maxDepth) for c in cams]
                rgb = torch.empty((V, h, w, 3), dtype=torch.uint8, device="cuda")

                def batch():
                    return rh.renderViews(base, cams, spp=spp, seeds=seeds, device=True)

                def renders():
                    ms = 0.0
                    for v in range(V):
                        ms += rh.render_device(jobs[v], rgb[v], spp=spp, seed=seeds[v])["ms_total"]
                    return ms

                try:
                    batch(), renders()  # warm-up
                except capi.RayHsError as e:
                    if e.code != capi.RH_ERR_OOM:
                        raise
                    res["runs"].append({"width": w, "height": h, "spp": spp, "views": V, "error": str(e),
                                        "free_gb": torch.cuda.mem_get_info()[0] / 1e9})
                    print(f"{w}x{h} {spp:2d} spp V={V:3d}: {e}", file=sys.stderr)
                    sc.close()
                    continue
                t_batch, t_renders, ms_batch, ms_renders = [], [], [], []
                for _ in range(a.reps):
                    t0 = time.perf_counter()
                    vs = batch()
                    t_batch.append((time.perf_counter() - t0) * 1e3)
                    ms_batch.append(vs.stats["ms_total"])
                    t0 = time.perf_counter()
                    ms_renders.append(renders())
                    t_renders.append((time.perf_counter() - t0) * 1e3)
                torch.cuda.synchronize()
                equal = bool(torch.equal(vs.pixels, rgb))
                max_diff = int((vs.pixels.int() - rgb.int()).abs().max().item())
                run = {"width": w, "height": h, "spp": spp, "views": V, "samples": V * w * h * spp,
                       "batch_ms": min(t_batch), "renders_ms": min(t_renders), "batch_ms_total": min(ms_batch),
                       "renders_ms_total": min(ms_renders), "batch_ms_all": t_batch, "renders_ms_all": t_renders,
                       "chunks": vs.stats["chunks"], "queue_factor": vs.stats["queue_factor"], "shadow_split": vs.stats["shadow_split"], "equal": equal, "max_diff": max_diff}
                run["speedup"] = run["renders_ms"] / run["batch_ms"]
                res["runs"].append(run)
                print(f"{w}x{h} {spp:2d} spp V={V:3d}: batch {run['batch_ms']:9.2f} ms, {V} renders {run['renders_ms']:9.2f} ms "
                      f"(x{run['speedup']:.2f}); equal {equal}", file=sys.stderr)
                del vs, rgb
                sc.close()
    line = json.dumps(res)
    print(line)
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
