"""Cost of the feature buffers (rh_render_features) on the bench view, beside rh_render of the same opts.

    python scripts/features_rate.py [--pack tests/golden/dragon_full.pack] [--width 3840 --height 2160] [--json out.json]

Workload: the bench scene and view at 3840 x 2160, RH_OFFSETS_SPLITMIX64 (seed 24), 1 spp and 16 spp, all four buffers
and no hit ids.  Per spp: the best of --reps timed calls after a warm-up call, each feature call followed by an rh_render
of the same opts, with device buffers (CUDA events around the call); then the same with host buffers (numpy outputs,
host clock around the call, which returns when they are written).  The card's name and power limit are read in the
same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import rayhs_b200 as rh  # noqa: E402
from scripts.ray_query_rate import card  # noqa: E402


def timed_device(fn) -> float:
    import torch

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def timed_host(fn) -> float:
    t0 = time.perf_counter()
    fn()
    return (time.perf_counter() - t0) * 1e3


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--pack", default=os.path.join(ROOT, "tests", "golden", "dragon_full.pack"))
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--spp", type=int, nargs="+", default=[1, 16])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--json", default=None, help="also write the result here")
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("features_rate.py measures on the GPU; no CUDA device here")
    sc = rh.Scene.from_pack(a.pack)
    job = rh.renderingFromScene(sc, a.width, a.height)
    rgb = torch.empty((a.height, a.width, 3), dtype=torch.uint8, device="cuda")
    res = {"card": card(), "pack": os.path.basename(a.pack), "width": a.width, "height": a.height, "runs": []}
    for spp in a.spp:
        def features(device):
            return lambda: rh.renderFeatures(job, spp=spp, seed=24, device=device)

        def render():
            rh.render_device(job, rgb, spp=spp, seed=24)

        run = {"spp": spp, "samples": a.width * a.height * spp}
        for device in (True, False):
            clock = timed_device if device else timed_host
            features(device)()  # warm-up: module load, scratch allocation
            render()
            feat, rend = [], []
            for _ in range(a.reps):
                feat.append(clock(features(device)))
                rend.append(clock(render))
            key = "device" if device else "host"
            run[key] = {"features_ms": min(feat), "render_ms": min(rend), "features_ms_all": feat, "render_ms_all": rend,
                        "mrays_s": run["samples"] / min(feat) / 1e3}
        res["runs"].append(run)
        print(f"{spp:3d} spp: features {run['device']['features_ms']:.2f} ms (device buffers), {run['host']['features_ms']:.2f} ms "
              f"(host buffers); render {run['device']['render_ms']:.2f} ms", file=sys.stderr)
    line = json.dumps(res)
    print(line)
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
