"""Adaptive sampling (rh_render_adaptive) on the bench view against uniform progressive sampling of the same stream.

    python scripts/adaptive_rate.py [--pack tests/golden/dragon_full.pack] [--width 3840 --height 2160] [--max-spp 64]
                                    [--batches 4,8] [--min-spp 8] [--thresholds 0.00196078,0.00784314] [--json out.json]

The view is the bench's: dragon_full at 3840x2160, SplitMix64 seed 24, device outputs.  Baseline: uniform progressive
sampling to --max-spp (progressiveRayTrace's loop, batch 8, RGB8 and linear outputs).  Adaptive: adaptiveRayTrace's loop
(AdaptiveAccumulator.add with the same batch until no pixel is active) for every --batches x --thresholds pair.
Reported per round: n_active, ms_total (CUDA events inside the library around the whole call) and, from a second run
with RH_FLAG_PROFILE, ms_resolve (the sinks, selection, commit and output kernels).  The selection and output kernels
are also timed on their own: a call with no active pixel runs only them (without outputs: the selection alone).  Per
run: samples traced, device time, and the error of the final image against the uniform --max-spp frame: the share of
pixels within 1 LSB in every channel, the share equal to the byte, and the linear RMSE.  The scene's renders are warmed
up first, so that its shadow-walk schedule is decided.  The card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

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
    ap.add_argument("--max-spp", type=int, default=64)
    ap.add_argument("--uniform-batch", type=int, default=8)
    ap.add_argument("--batches", default="4,8")
    ap.add_argument("--min-spp", type=int, default=8)
    ap.add_argument("--thresholds", default=f"{0.5 / 255:.8f},{2 / 255:.8f}")
    ap.add_argument("--seed", type=int, default=24)
    ap.add_argument("--json", default=None, help="also write the result here")
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("adaptive_rate.py measures on the GPU; no CUDA device here")
    sc = rh.Scene.from_pack(a.pack)
    job = rh.renderingFromScene(sc, a.width, a.height)
    W, H, S = a.width, a.height, a.max_spp
    res = {"card": card(), "pack": os.path.basename(a.pack), "width": W, "height": H, "max_spp": S, "min_spp": a.min_spp,
           "seed": a.seed, "outputs": "device RGB8 + linear"}
    frame = torch.empty((H, W, 3), dtype=torch.uint8, device="cuda")
    for _ in range(4):  # the scene's timing frames: afterwards its shadow-walk schedule is decided
        rh.render_device(job, frame, spp=16, seed=a.seed)

    # uniform baseline: every pixel gets every sample of the stream
    acc = rh.Accumulator(job, stream_spp=S, device=True)
    for rep in range(2):  # (the first pass is a warm-up)
        acc.reset()
        ms = []
        for _ in range(S // a.uniform_batch):
            img = acc.add(a.uniform_batch, seed=a.seed)
            ms.append(img.stats["ms_total"])
    ref_px, ref_lin = img.pixels, img.linear
    res["uniform"] = {"batch": a.uniform_batch, "calls": len(ms), "samples": W * H * S, "ms_total_per_call": ms,
                      "ms_total_sum": sum(ms)}
    acc.close()
    print(f"uniform {S} spp in batches of {a.uniform_batch}: {sum(ms):.1f} ms", file=sys.stderr)

    def adaptive(ad, batch, threshold, profile=False):
        ad.reset()
        rounds = []
        while True:
            img = ad.add(batch, a.seed, threshold, min_spp=a.min_spp, profile=profile)
            st = img.stats
            rounds.append({"n_active": st["n_active"], "ms_total": st["ms_total"], "ms_resolve": st["ms_resolve"],
                           "chunks": st["chunks"]})
            if st["n_active"] == 0:
                return rounds, img

    res["adaptive"] = []
    for batch in (int(b) for b in a.batches.split(",")):
        for threshold in (float(t) for t in a.thresholds.split(",")):
            ad = rh.AdaptiveAccumulator(job, S, device=True)
            adaptive(ad, batch, threshold)  # warm-up
            rounds, img = adaptive(ad, batch, threshold)
            prof, pimg = adaptive(ad, batch, threshold, profile=True)
            same = bool(torch.equal(pimg.pixels, img.pixels))
            # the selection and output kernels alone: the state has converged, so a call traces nothing
            idle = ad.add(batch, a.seed, threshold, min_spp=a.min_spp, profile=True).stats
            bare = ad.add(batch, a.seed, threshold, min_spp=a.min_spp, profile=True, rgb=False, linear=False).stats
            counts = ad.state()[0].to(torch.int64)
            d = (img.pixels.to(torch.int16) - ref_px.to(torch.int16)).abs().amax(dim=-1)
            rmse = float(torch.sqrt(((img.linear - ref_lin) ** 2).mean()))
            traced = sum(r["n_active"] for r in rounds) * batch
            run = {"batch": batch, "threshold": threshold, "rounds": rounds[:-1], "idle_round": rounds[-1],
                   "profiled_ms_resolve": [r["ms_resolve"] for r in prof],
                   "select_ms": bare["ms_resolve"], "select_output_ms": idle["ms_resolve"],
                   "output_ms": idle["ms_resolve"] - bare["ms_resolve"],
                   "samples": traced, "samples_share_of_uniform": traced / (W * H * S),
                   "ms_total_sum": sum(r["ms_total"] for r in rounds),
                   "mean_spp": float(counts.float().mean()), "pixels_at_max_spp": float((counts == S).float().mean()),
                   "within_1_lsb": float((d <= 1).float().mean()), "equal_bytes": float((d == 0).float().mean()),
                   "max_lsb": int(d.max()), "linear_rmse": rmse, "profiled_run_same_bytes": same}
            res["adaptive"].append(run)
            ad.close()
            print(f"batch {batch} threshold {threshold:.6f}: {len(rounds) - 1} rounds, n_active {[r['n_active'] for r in rounds]}, "
                  f"{traced / (W * H * S) * 100:.1f} % of the samples, {run['ms_total_sum']:.1f} ms "
                  f"(uniform {sum(ms):.1f}); select {run['select_ms']:.3f} ms, output {run['output_ms']:.3f} ms; "
                  f"within 1 LSB {run['within_1_lsb'] * 100:.3f} %, RMSE {rmse:.2e}", file=sys.stderr)
    line = json.dumps(res)
    print(line)
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            f.write(line + "\n")
    return 0 if all(r["profiled_run_same_bytes"] for r in res["adaptive"]) else 1


if __name__ == "__main__":
    sys.exit(main())
