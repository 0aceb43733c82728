"""Cost of progressive rendering (rh_render_accumulate) on the bench view, beside one rh_render of the same samples.

    python scripts/progressive_rate.py [--pack tests/golden/dragon_full.pack] [--width 3840 --height 2160] [--spp 16]
                                       [--batches 1,2,4,8,16] [--reps 3] [--json out.json]

The view is the bench's: dragon_full at 3840x2160, SplitMix64 seed 24, device outputs.  One rh_render of --spp samples is
compared with the same samples through an accumulator in batches of 1, 2, 4, 8 and 16 samples per call, each call
writing RGB8 and the linear colours.  Reported per batch size: each call's ms_total (CUDA events inside the library
around the call's device work) and host time (the call returns when its outputs are written), their sums over the
frame, and — in separate runs with RH_FLAG_PROFILE, which times every launch on its own — the sink kernel's time
(ms_resolve: accumulate_resolve_kernel) against resolve_kernel's in the one-shot render.  Timings are the best of --reps
frames after a warm-up frame; the scene's renders are warmed up first, so that its shadow-walk schedule is decided.
The final bytes of every accumulated frame are checked against the one-shot frame.  The card's name and power limit
are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import rayhs_b200 as rh  # noqa: E402
from ray_query_rate import card  # noqa: E402


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--pack", default=os.path.join(ROOT, "tests", "golden", "dragon_full.pack"))
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--spp", type=int, default=16)
    ap.add_argument("--seed", type=int, default=24)
    ap.add_argument("--batches", default="1,2,4,8,16")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--json", default=None, help="also write the result here")
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("progressive_rate.py measures on the GPU; no CUDA device here")
    batches = [int(b) for b in a.batches.split(",")]
    if any(b < 1 or a.spp % b for b in batches):
        sys.exit(f"every batch must divide --spp {a.spp}")
    sc = rh.Scene.from_pack(a.pack)
    job = rh.renderingFromScene(sc, a.width, a.height)
    res = {"card": card(), "pack": os.path.basename(a.pack), "width": a.width, "height": a.height, "spp": a.spp,
           "seed": a.seed, "outputs": "device RGB8 + linear"}

    one = torch.empty((a.height, a.width, 3), dtype=torch.uint8, device="cuda")
    for _ in range(4):  # the scene's timing frames: afterwards its shadow-walk schedule is decided
        rh.render_device(job, one, spp=a.spp, seed=a.seed)

    def one_shot(profile=False):
        t0 = time.perf_counter()
        st = rh.render_device(job, one, spp=a.spp, seed=a.seed, profile=profile)
        return (time.perf_counter() - t0) * 1e3, st

    def frame(acc, batch, profile=False):
        """One frame of --spp samples in calls of `batch`: per-call (host ms, stats) and the last image."""
        acc.reset()
        calls = []
        for _ in range(a.spp // batch):
            t0 = time.perf_counter()
            img = acc.add(batch, seed=a.seed, profile=profile)
            calls.append(((time.perf_counter() - t0) * 1e3, img.stats))
        return calls, img

    one_shot()
    runs = [one_shot() for _ in range(a.reps)]
    best = min(runs, key=lambda r: r[1]["ms_total"])
    prof = one_shot(profile=True)[1]
    res["one_shot"] = {"ms_total": best[1]["ms_total"], "host_ms": best[0], "ms_total_all": [r[1]["ms_total"] for r in runs],
                       "chunks": best[1]["chunks"], "resolve_kernel_ms": prof["ms_resolve"]}
    want = one.clone()

    res["batches"] = {}
    for b in batches:
        acc = rh.Accumulator(job, stream_spp=a.spp, device=True)
        frame(acc, b)  # warm-up
        frames = [frame(acc, b) for _ in range(a.reps)]
        calls, img = min(frames, key=lambda f: sum(st["ms_total"] for _, st in f[0]))
        same = bool(torch.equal(img.pixels, want))
        pcalls, pimg = frame(acc, b, profile=True)
        same = same and bool(torch.equal(pimg.pixels, want))
        res["batches"][str(b)] = {
            "calls": len(calls),
            "ms_total_per_call": [st["ms_total"] for _, st in calls],
            "host_ms_per_call": [ms for ms, _ in calls],
            "ms_total_sum": sum(st["ms_total"] for _, st in calls),
            "host_ms_sum": sum(ms for ms, _ in calls),
            "ms_total_sum_all": [sum(st["ms_total"] for _, st in f[0]) for f in frames],
            "sink_ms_per_call": [st["ms_resolve"] for _, st in pcalls],
            "sink_ms_mean": sum(st["ms_resolve"] for _, st in pcalls) / len(pcalls),
            "final_bytes_equal_one_shot": same,
        }
        acc.close()
        del img, pimg
        print(f"batch {b:2d}: {len(calls):2d} calls, ms_total sum {res['batches'][str(b)]['ms_total_sum']:.2f} "
              f"(one-shot {res['one_shot']['ms_total']:.2f}), sink {res['batches'][str(b)]['sink_ms_mean']:.3f} ms/call "
              f"(resolve_kernel {prof['ms_resolve']:.3f}), bytes equal: {same}", file=sys.stderr)
    line = json.dumps(res)
    print(line)
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            f.write(line + "\n")
    return 0 if all(v["final_bytes_equal_one_shot"] for v in res["batches"].values()) else 1


if __name__ == "__main__":
    sys.exit(main())
