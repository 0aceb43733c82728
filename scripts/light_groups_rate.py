"""Cost of the light groups (rh_render_light_groups) on the bench view, beside rh_render and beside the workaround of
one render per light plus one with every light off.

    python scripts/light_groups_rate.py [--pack tests/golden/dragon_full.pack] [--width 3840 --height 2160] [--json out.json]

Workload: the bench scene and view at 3840 x 2160, RH_OFFSETS_SPLITMIX64 (seed 24), 16 spp and 1 spp, device outputs.
Per spp, after a warm-up round (which also settles the scene's shadow schedule), --reps rounds alternate four calls:
rh_render; light groups with one group holding every light; light groups with one group per light; and the workaround
(L + 1 renders, each after a colours-only Scene.update that zeroes every light but one, or all of them).  Each call's
ms_total (device time of the frame, from rh_stats) is kept, the best of the rounds reported; the workaround's is the sum
of its renders (its updates, host work of a few tens of microseconds, are not counted).  Also recorded: chunks, and from
separate RH_FLAG_PROFILE runs ms_shadow and ms_resolve.  The card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import rayhs_b200 as rh  # noqa: E402
from scripts.ray_query_rate import card  # noqa: E402


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--pack", default=os.path.join(ROOT, "tests", "golden", "dragon_full.pack"))
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--spp", type=int, nargs="+", default=[16, 1])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--json", default=None, help="also write the result here")
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("light_groups_rate.py measures on the GPU; no CUDA device here")
    sc = rh.Scene.from_pack(a.pack)
    job = rh.renderingFromScene(sc, a.width, a.height)
    lights = sc.lights
    L = len(lights)
    rgb = torch.empty((a.height, a.width, 3), dtype=torch.uint8, device="cuda")
    res = {"card": card(), "pack": os.path.basename(a.pack), "width": a.width, "height": a.height, "lights": L, "runs": []}

    def only(keep):
        """Colours-only update: every light but those in `keep` black."""
        t = (type(lights))(*lights)  # (a copy of the original table)
        for l in range(L):
            if l not in keep:
                t[l].color[0] = t[l].color[1] = t[l].color[2] = 0.0
        info = sc.update(lights=t)
        assert info["colours_only"] == 1, info

    for spp in a.spp:
        calls = {
            "render": lambda: rh.render_device(job, rgb, spp=spp, seed=24),
            "groups_1": lambda: rh.renderLightGroups(job, spp=spp, seed=24, groups=[0] * L, device=True).stats,
            f"groups_{L}": lambda: rh.renderLightGroups(job, spp=spp, seed=24, device=True).stats,
        }

        def workaround():
            ms, chunks = 0.0, 0
            for keep in [[l] for l in range(L)] + [[]]:
                only(keep)
                st = rh.render_device(job, rgb, spp=spp, seed=24)
                ms += st["ms_total"]
                chunks = max(chunks, st["chunks"])
            sc.update(lights=lights)
            return {"ms_total": ms, "chunks": chunks}

        calls[f"workaround_{L + 1}_renders"] = workaround
        for _ in range(4):  # warm-up: module load, scratch, and the render's shadow-schedule timing frames
            for fn in calls.values():
                fn()
        times = {k: [] for k in calls}
        chunks = {}
        for _ in range(a.reps):
            for k, fn in calls.items():
                st = fn()
                times[k].append(st["ms_total"])
                chunks[k] = st["chunks"]
        run = {"spp": spp, "samples": a.width * a.height * spp, "shadow_split": rh.render_device(job, rgb, spp=spp, seed=24)["shadow_split"]}
        for k in calls:
            run[k] = {"ms_total": min(times[k]), "ms_total_all": times[k], "chunks": chunks[k]}
        prof = {"render": rh.render(job, spp=spp, seed=24, profile=True).stats,
                "groups_1": rh.renderLightGroups(job, spp=spp, seed=24, groups=[0] * L, device=True, profile=True).stats,
                f"groups_{L}": rh.renderLightGroups(job, spp=spp, seed=24, device=True, profile=True).stats}
        for k, st in prof.items():
            run[k].update(ms_shadow=st["ms_shadow"], ms_resolve=st["ms_resolve"], ms_trace=st["ms_trace"], profile_chunks=st["chunks"])
        res["runs"].append(run)
        print(f"{spp:3d} spp: " + ", ".join(f"{k} {run[k]['ms_total']:.2f} ms ({run[k]['chunks']} chunks)" for k in calls), file=sys.stderr)
    line = json.dumps(res)
    print(line)
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
