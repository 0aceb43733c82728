#!/usr/bin/env python
"""bench.py — Mrays/s of the RayHs ray-casting path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c4|c5] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step = one frame of the workload.  Default workload "c4": dragon.json with the full-res dragon.obj at
3840x2160, 16 samples per pixel, maxDepth 3 (BASELINE.json configs[3], the configuration the metric is quoted
on; it fits one GPU).  "c5": BASELINE.json configs[4], the synthetic stress scene — 10 M random triangles +
1 000 spheres at 7680x4320, 64 spp (SURVEY 8d); run it with --gpus 1/2/4/8.  Rays = closestIntersection +
shadowIntersection calls (SURVEY.md 8d), counted by the kernels; the same count comes out of the oracle.

  value  frame rendered with the sample offsets already in HBM (c5: regenerated on the device from the stream's
         seed — the full stream is 34 GB) and the RGB8 frame left in HBM
  e2e    the same frame through rh_render with HOST buffers: pinned f64 offsets in (H2D, overlapped chunk by
         chunk), RGB8 frame out (D2H), all inside the timed region
N > 1: one process per GPU, scene replicated, image rows sharded as interleaved bands, frame assembled by peer
stores over NVLink or one NCCL all-gather + rh_deinterleave_bands (inside the timed region); the frame is fixed,
so "scaling": "strong".

parity: the frame the timed steps rendered against the oracle (oracle/oracle.cpp, the CPU restatement of the
reference) — c4: every row the cpu_baseline leg renders (all 2160 when the host is fast enough); c5: 16 rows x
64 columns x 64 spp; hit ids and RGB8 bytes.

--dump-outputs DIR: what the last timed step computed, as float32/float64 .npy files in DIR (at most 64 MB) — rgb.npy
  [n, width, 3], the RGB8 values of n rows of the complete frame (all rows when they fit 48 MB as float32, else a fixed
  seeded sample), rgb_rows.npy the indices of those rows, rays_by_class.npy [5] the frame's primary, reflect, probe,
  exit and shadow ray counts.  The inputs are seeded, so two builds run with the same arguments can be compared file
  for file.

--impl reference times the reference's own CPU algorithm (the C++ restatement in oracle/, because GHC is not in
this image: kind "port") with all host threads on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

T_PROCESS_START = time.time()
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "c4": dict(pack="dragon_full", width=3840, height=2160, spp=16, seed=24, steps=5,
               metric="Mrays/s (primary + secondary + shadow), dragon.json full-res at 3840x2160, 16 spp",
               desc="dragon.json + dragon.obj (27228 tris), {w}x{h}, {spp} spp, maxDepth 3, 3 point lights (BASELINE.json configs[3])",
               data="synthetic sample offsets (SplitMix64 seed 24); shipped dragon.obj scene"),
    "c5": dict(tris=10_000_000, spheres=1000, width=7680, height=4320, spp=64, seed=24, steps=2,
               metric="Mrays/s (primary + secondary + shadow), synthetic stress scene (10 M triangles + 1 k spheres) at 7680x4320, 64 spp",
               desc="synthetic stress scene: {tris} random triangles + {spheres} spheres + checker floor, {w}x{h}, {spp} spp, maxDepth 3, "
                    "3 point lights (BASELINE.json configs[4], SURVEY 8d C5)",
               data="synthetic scene (SplitMix64 seed 0x5EED) and synthetic sample offsets (SplitMix64 seed 24)"),
}


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        if os.environ.get("RAYHS_BENCH_NO_SMI"):   # (diagnosis only: how much the polling itself costs)
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.t.join(timeout=2)
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def algorithmic_bytes(st: dict, offset_bytes: int, tables_in_smem: bool, n_pixels: int, spp: int) -> dict:
    """DESIGN.md 5: per kernel and frame, from the instrumented (RH_FLAG_COUNT) kernels' own counters, two kinds of bytes.
    `stream`: bytes that must cross HBM — sample offsets, queue entries written and read (ray 64 B, hit 88 B, queued
    hit 92 B, + the point re-read per walked pair 32 B), accumulator updates (24 B): GBs per frame, read or written once.
    `gather`: record fetches an SM issues — node records beyond the shared-memory-staged top levels (64 B) and triangle
    records (80 B), both counted once per warp instruction (lanes reading the same record share one fetch), winning
    shading records (128 B), texels (24 B), object records of sphere-tree leaves when the object table is not staged
    (96 B).  Gathers are served by L1, L2 or HBM: of them only min(gather, the record set's size per launch) HAS to
    cross HBM (`hbm_compulsory`, formed by the caller).  The occluder, light and material tables and the top tree
    levels live in shared memory and are not traffic."""
    prim = 0 if tables_in_smem else 96
    out = {
        "trace": {"stream": offset_bytes * st["rays_primary"] + 2 * 64 * st["queued_rays"] + 88 * st["shadow_tasks"],
                  "gather": 64 * st["node_visits_global"] + 80 * st["tri_records"] + prim * st["prim_tests"] + 128 * st["shade_fetches"]
                            + 24 * st["texel_fetches"]},
        "classify": {"stream": 88 * st["shadow_tasks"] + 92 * st["shadow_tasks_queued"] + 24 * (st["shadow_tasks"] - st["shadow_tasks_queued"]),
                     "gather": 0},
        "walk": {"stream": 92 * st["shadow_tasks_queued"] + 32 * st["shadow_walk_pairs"] + 24 * st["shadow_tasks_queued"],
                 "gather": 64 * st["shadow_node_visits_global"] + 80 * st["shadow_tri_records"] + prim * st["shadow_prim_tests"]},
        "resolve": {"stream": (24 * spp + 3) * n_pixels, "gather": 0},
    }
    return out


def compare_u8(a: np.ndarray, b: np.ndarray) -> dict:
    d = np.abs(a.astype(np.int32) - b.astype(np.int32))
    mse = float((d.astype(np.float64) ** 2).mean()) if d.size else 0.0
    return {"exact": float((d == 0).mean()) if d.size else 1.0, "within1": float((d <= 1).mean()) if d.size else 1.0,
            "max_diff": int(d.max()) if d.size else 0, "psnr": (float("inf") if mse == 0 else 10 * np.log10(255.0 ** 2 / mse))}


def c4_oracle_sample(sc, W, H, spp, offsets, seconds_target, threads=0, want_ids=False):
    """Reference algorithm (oracle port) on every k-th row of the frame; returns (Mrays/s, description, result, rows)."""
    from oracle.orc import OracleScene

    o = OracleScene(sc.raw)
    probe_step = max(1, H // 8)
    r = o.render(sc.camera, W, H, sc.max_depth, spp=spp, offsets=offsets, rows=(0, H, probe_step), threads=threads, want_ids=False)
    rate = r["rays_total"] / max(r["seconds"], 1e-9)
    rows_probe = len(range(0, H, probe_step))
    rays_per_row = r["rays_total"] / rows_probe
    n_rows = int(max(rows_probe, min(H, seconds_target * rate / rays_per_row)))
    step = max(1, H // n_rows)
    r = o.render(sc.camera, W, H, sc.max_depth, spp=spp, offsets=offsets, rows=(step // 2, H, step), threads=threads, want_ids=want_ids)
    rows = np.arange(step // 2, H, step)
    o.close()
    return (r["rays_total"] / r["seconds"] / 1e6,
            f"{len(rows)} of {H} rows (every {step}th) of the {W}x{H}x{spp}spp frame, {r['seconds']:.1f} s", r, rows)


C5_ROWS, C5_COLS = 16, 64   # parity / CPU-baseline sample of the c5 frame: 16 rows x 64 columns x 64 spp


def c5_sample_grid(W, H):
    rstep, cstep = H // C5_ROWS, W // C5_COLS
    return (rstep // 2 + 7, H, rstep), (cstep // 2 + 3, W, cstep)


def c5_oracle_sample(sc, W, H, spp, seed, rows, cols, threads=0):
    from oracle.orc import OracleScene

    t0 = time.time()
    o = OracleScene(sc.raw)
    build_s = time.time() - t0
    r = o.render_sample(sc.camera, W, H, sc.max_depth, spp=spp, seed=seed, rows=rows, cols=cols, threads=threads)
    o.close()
    n = len(r["rows"]) * len(r["cols"])
    return (r["rays_total"] / r["seconds"] / 1e6,
            f"{len(r['rows'])} rows x {len(r['cols'])} columns x {spp} spp = {n * spp} pixel samples of the {W}x{H} frame, "
            f"{r['seconds']:.1f} s (+ {build_s:.0f} s for the oracle's own single-threaded tree build, not timed)", r)


RAY_CLASSES = ("rays_primary", "rays_reflect", "rays_probe", "rays_exit", "rays_shadow")
DUMP_FRAME_BYTES = 48_000_000   # --dump-outputs: the frame's share of the 64 MB the dump may take


def dump_rows(H: int, W: int) -> np.ndarray:
    """Rows of the frame --dump-outputs writes: all of them if they fit DUMP_FRAME_BYTES as float32, else a sorted
    sample drawn with a fixed seed (the same rows in every run of the same frame size)."""
    n = min(H, DUMP_FRAME_BYTES // (W * 3 * 4))
    if n == H:
        return np.arange(H)
    return np.sort(np.random.default_rng(0).choice(H, n, replace=False))


def dump_outputs(path: str, rgb_rows: np.ndarray, rows: np.ndarray, rays_by_class: np.ndarray) -> None:
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "rgb.npy"), rgb_rows.astype(np.float32))
    np.save(os.path.join(path, "rgb_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(path, "rays_by_class.npy"), rays_by_class.astype(np.float64))


def make_scene(rh, wl):
    if "pack" in wl:
        return rh.Scene.from_pack(os.path.join(ROOT, "tests", "golden", wl["pack"] + ".pack"))
    return rh.Scene.synthetic(wl["tris"], wl["spheres"])


def config_dict(wl, n_gpus, name):
    w, h, spp = wl["width"], wl["height"], wl["spp"]
    offs = (f"per-pixel f64 pairs, RandomSamples.hs shape, host-generated ({w * h * spp * 16 / 1e9:.1f} GB per frame)" if name == "c4" else
            f"per-pixel f64 pairs, RandomSamples.hs shape ({w * h * spp * 16 / 1e9:.1f} GB per frame): `value` regenerates the stream on the "
            f"device from its seed, `e2e` uploads every rank's rows from pinned host memory")
    return {"workload": wl["desc"].format(w=w, h=h, spp=spp, tris=wl.get("tris"), spheres=wl.get("spheres")),
            "offsets": offs, "parallelism": f"rows{n_gpus}" if n_gpus > 1 else "1gpu",
            "l2": "inputs larger than L2: the sample offsets and the ray / hit queues (GBs per frame) stream through; "
                  + ("the 4.6 MB scene is L2-resident by design" if name == "c4" else "the 2.1 GB scene exceeds the 126 MB L2")}


def run_reference(args, rank, world, wl, name):
    if rank != 0:
        return
    W, H, spp = wl["width"], wl["height"], wl["spp"]
    if name == "c4":
        # nothing of the product on this arm: the pack is read and the offset stream generated by oracle/packio.py
        from oracle import packio

        sc = packio.PackScene(os.path.join(ROOT, "tests", "golden", wl["pack"] + ".pack"))
    else:
        import rayhs_b200 as rh   # (the synthetic scene generator is the front end's: rh_make_synthetic)

        sc = make_scene(rh, wl)
    cores = os.cpu_count() or 1
    per_step = max(2.0, min(20.0, 150.0 / max(1, args.steps + args.warmup)))
    vals, sample = [], ""
    t0 = time.time()
    if name == "c4":
        offsets = packio.sample_offsets(W * H, spp, wl["seed"])
        for i in range(args.warmup + args.steps):
            v, sample, _, _ = c4_oracle_sample(sc, W, H, spp, offsets, per_step)
            if i >= args.warmup:
                vals.append(v)
    else:
        from oracle.orc import OracleScene

        o = OracleScene(sc.raw)   # (one tree build for all steps)
        rows, cols = c5_sample_grid(W, H)
        t0 = time.time()
        for i in range(args.warmup + args.steps):
            r = o.render_sample(sc.camera, W, H, sc.max_depth, spp=max(1, spp // 8), seed=wl["seed"], rows=rows, cols=cols, want_ids=False)
            if i >= args.warmup:
                vals.append(r["rays_total"] / r["seconds"] / 1e6)
            sample = f"{len(r['rows'])} rows x {len(r['cols'])} columns x {max(1, spp // 8)} spp of the {W}x{H} frame, {r['seconds']:.1f} s per step"
        o.close()
    value = float(np.mean(vals))
    ms = 1e3 * (time.time() - t0) / max(1, args.warmup + args.steps)
    line = {"impl": "reference", "metric": wl["metric"], "value": value, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": wl["data"], "config": config_dict(wl, 1, name),
            "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "C++ restatement of the reference algorithm (oracle/oracle.cpp: un-pruned traversal, per-object linear scan, "
                    "full closest-hit shadow queries, double), all host threads; GHC is not installed on this image"}
    print(json.dumps(line), flush=True)


def cold_start(name: str, wl: dict) -> dict | None:
    """One-shot use, like the reference CLI (RayHs.hs:215-234): a fresh process loads the scene, initialises the library,
    uploads the scene and renders ONE frame (no warm-up, no tuning frames) to host memory.  Wall times in ms."""
    code = r'''
import json, os, sys, time
t0 = time.time()
sys.path.insert(0, %r)
import numpy as np
import rayhs_b200 as rh
from rayhs_b200 import capi
t1 = time.time()
rh.init(0)
t2 = time.time()
wl = %r
sc = rh.Scene.from_pack(os.path.join(%r, "tests", "golden", wl["pack"] + ".pack")) if "pack" in wl else rh.Scene.synthetic(wl["tris"], wl["spheres"])
_ = sc.flat
t3 = time.time()
_ = sc.device
t4 = time.time()
job = rh.renderingFromScene(sc, wl["width"], wl["height"])
img = rh.render(job, spp=wl["spp"], seed=wl["seed"], shadow="pooled")
t5 = time.time()
setup = rh.scene_setup_ms(sc)
print(json.dumps({"import_ms": 1e3 * (t1 - t0), "rh_init_ms": 1e3 * (t2 - t1), "scene_load_and_flatten_ms": 1e3 * (t3 - t2),
                  "rh_scene_create_ms": 1e3 * (t4 - t3), "first_frame_ms": 1e3 * (t5 - t4), "total_ms": 1e3 * (t5 - t0),
                  "rh_scene_create_split_ms": setup, "first_frame_device_ms": img.stats["ms_total"]}))
''' % (ROOT, {k: v for k, v in wl.items() if k in ("pack", "tris", "spheres", "width", "height", "spp", "seed")}, ROOT)
    try:
        t0 = time.time()
        r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900)
        wall = 1e3 * (time.time() - t0)
        d = json.loads(r.stdout.strip().splitlines()[-1])
        d["process_wall_ms"] = wall
        d["note"] = ("fresh process: import (ctypes only) + rh_init (CUDA context) + scene load/flatten on the host + rh_scene_create + one "
                     "frame with device-generated offsets, RGB8 on the host; no warm-up frame")
        return d
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)[:200]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default: the workload's)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cold-start", action="store_true")
    ap.add_argument("--width", type=int, default=0, help="override (debug only; the reported config changes with it)")
    ap.add_argument("--height", type=int, default=0)
    ap.add_argument("--spp", type=int, default=0)
    ap.add_argument("--tris", type=int, default=0)
    ap.add_argument("--band-height", type=int, default=0, help="rows per interleaved band at N > 1 (default: the library's choice)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    name = args.workload
    wl = dict(WORKLOADS[name])
    for k in ("width", "height", "spp", "tris"):
        if getattr(args, k):
            wl[k] = getattr(args, k)
    if args.steps is None:
        args.steps = wl["steps"]
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the frame of the product path; the reference arm renders a timing-dependent row sample")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world, wl, name)
        return
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist

    import rayhs_b200 as rh
    from rayhs_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    # stdout carries exactly one JSON line: anything a library prints to fd 1 in between (NCCL's version banner under
    # NCCL_DEBUG=VERSION ignores NCCL_DEBUG_FILE) goes to stderr; fd 1 is restored for the final print
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    # one-shot use first, while this process holds no device memory: a fresh process renders one frame
    cold = cold_start(name, wl) if (rank == 0 and world == 1 and not args.no_cold_start) else None
    t0 = time.time()
    rh.init(local_rank)
    t_init = time.time() - t0
    L = capi.lib()
    W, H, spp, seed = wl["width"], wl["height"], wl["spp"], wl["seed"]
    t0 = time.time()
    sc = make_scene(rh, wl)
    _ = sc.flat
    t_host = time.time() - t0
    t0 = time.time()
    _ = sc.device
    t_create = time.time() - t0
    setup = {"rh_init_ms": 1e3 * t_init, "scene_load_and_flatten_ms": 1e3 * t_host, "rh_scene_create_ms": 1e3 * t_create,
             "rh_scene_create_split_ms": rh.scene_setup_ms(sc),
             "note": "outside the timed steps; scene_load_and_flatten = front end on the host (pack read or synthetic generator, then the "
                     "KDTree.hs:68-90 build + flattening a Haskell host would do); rh_scene_create = the library's own set-up"}
    job = rh.renderingFromScene(sc, W, H)
    G = world
    bh = args.band_height or L.rh_default_band_height(H, G)
    rows = L.rh_shard_rows(H, G, bh)
    row_samples = W * spp
    c5 = name != "c4"

    # host inputs.  c4: the full-frame offset stream, pinned (what the Haskell host would hand over).  c5: only this
    # rank's rows of the stream (34 GB in full), shard-compact, generated band by band from the counter-based generator.
    if not c5:
        off_host = torch.empty((W * H, spp, 2), dtype=torch.float64, pin_memory=True)
        L.rh_sample_offsets_f64(seed, W * H, spp, off_host.data_ptr())
        off_dev = off_host.cuda()
    else:
        try:
            off_host = torch.empty((rows * W, spp, 2), dtype=torch.float64, pin_memory=True)
        except RuntimeError:   # (34 GB of pinned memory at N = 1)
            off_host = torch.empty((rows * W, spp, 2), dtype=torch.float64)
        for lb in range(rows // bh):
            grow = (lb * G + rank) * bh
            n = max(0, min(bh, H - grow))
            if n:
                L.rh_sample_offsets_f64_at(seed, grow * W, n * W, spp, off_host.data_ptr() + lb * bh * row_samples * 16)
        off_dev = None
    rgb_dev = torch.empty((rows, W, 3), dtype=torch.uint8, device="cuda")
    gathered = torch.empty((G, rows, W, 3), dtype=torch.uint8, device="cuda") if G > 1 else None
    full_dev = torch.empty((H, W, 3), dtype=torch.uint8, device="cuda") if G > 1 else None
    rgb_host = torch.empty((rows, W, 3), dtype=torch.uint8, pin_memory=True)
    full_host = torch.empty((H, W, 3), dtype=torch.uint8, pin_memory=True)

    def assemble():
        if G > 1:
            dist.all_gather_into_tensor(gathered, rgb_dev)
            torch.cuda.current_stream().synchronize()
            capi.check(L.rh_deinterleave_bands(gathered.data_ptr(), full_dev.data_ptr(), W, H, G, bh))

    # N > 1, fused exchange: every rank's resolve kernel stores its rows straight into all ranks' full frames (CUDA IPC
    # mappings, NVLink peer stores); one barrier after the render call completes the frame everywhere.
    peers = rh.PeerFrames(H, W) if G > 1 else None
    dev_kw = dict(seed=seed) if c5 else dict(offsets_dev=off_dev)
    host_kw = dict(offsets_dev=off_host, shard_offsets=True) if c5 else dict(offsets_dev=off_host)

    def step_device_nccl(**kw):
        st = rh.render_device(job, rgb_dev, spp=spp, shard_index=rank, shard_count=G, band_height=bh, **dev_kw, **kw)
        assemble()
        return st

    def step_device_fused(**kw):
        st = rh.render_device(job, None, spp=spp, shard_index=rank, shard_count=G, band_height=bh, peer_frames=peers.pointers, **dev_kw, **kw)
        dist.barrier()
        return st

    def step_device(**kw):
        if G == 1:
            return rh.render_device(job, rgb_dev, spp=spp, **dev_kw, **kw)
        return step_device_fused(**kw) if use_fused[0] else step_device_nccl(**kw)

    def step_e2e():
        if G == 1 and not c5:
            # the call a host makes: rh_render with host buffers in and out (pinned offsets in, RGB8 frame out)
            return rh.render(job, spp=spp, offsets=off_host, out=rgb_host.numpy()).stats
        if G == 1:
            st = rh.render_device(job, rgb_dev, spp=spp, **host_kw)
            rgb_host.copy_(rgb_dev)
            return st
        if use_fused[0]:
            st = rh.render_device(job, None, spp=spp, shard_index=rank, shard_count=G, band_height=bh, peer_frames=peers.pointers, **host_kw)
            dist.barrier()
            full_host.copy_(peers.frame)
            return st
        st = rh.render_device(job, rgb_dev, spp=spp, shard_index=rank, shard_count=G, band_height=bh, **host_kw)
        assemble()
        full_host.copy_(full_dev)
        return st

    use_fused = [G > 1]

    def barrier():
        if G > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        stats = [fn() for _ in range(k)]
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if G > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item() / k, stats

    def total_rays(st):
        r = torch.tensor([st["rays_primary"] + st["rays_reflect"] + st["rays_probe"] + st["rays_exit"] + st["rays_shadow"]],
                         dtype=torch.float64, device="cuda")
        if G > 1:
            dist.all_reduce(r, op=dist.ReduceOp.SUM)
        return r.item()

    # warm-up (also sizes the library's scratch buffers and lets the library time its two shadow-walk schedules)
    for _ in range(args.warmup):
        step_device()
    # (e2e: the streamed frame plans its chunks from the previous frame's measured row costs, and the first frame with
    # the new plan re-sizes its scratch: three untimed frames, like the device arm)
    for _ in range(max(3, args.warmup) if not c5 else 1):
        step_e2e()

    # N > 1: time both exchanges, report the frame with the faster one (both are in the JSON line)
    exchange = None
    if G > 1:
        step_device_nccl()
        ms_nccl, _ = timed(step_device_nccl, args.steps)
        ms_fused, _ = timed(step_device_fused, args.steps)
        use_fused[0] = ms_fused <= ms_nccl
        exchange = {"used": "peer_stores" if use_fused[0] else "nccl_allgather", "ms_per_step_peer_stores": ms_fused,
                    "ms_per_step_nccl_allgather": ms_nccl,
                    "note": "peer_stores: resolve kernel writes finished rows into every rank's frame over NVLink (CUDA IPC), "
                            "then one barrier; nccl_allgather: compact bands -> all_gather_into_tensor -> rh_deinterleave_bands"}

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = L.rh_launch_count()
    ms_dev, stats = timed(step_device, args.steps)
    launches = (L.rh_launch_count() - launches0) // args.steps
    dumped = None
    if args.dump_outputs and rank == 0:   # the last timed step's frame, before the calls below render into it again
        dump_idx = dump_rows(H, W)
        frame = rgb_dev if G == 1 else (peers.frame if use_fused[0] else full_dev)
        dumped = frame[torch.from_numpy(dump_idx).cuda()].cpu().numpy()
    ms_e2e, stats_e2e = timed(step_e2e, args.steps)
    ms_seeded = None
    if G == 1 and not c5:  # beside e2e: the same call with the offset stream regenerated on the device from its seed (no upload)
        seeded = lambda: rh.render(job, spp=spp, seed=seed, out=rgb_host.numpy()).stats
        seeded()
        ms_seeded, _ = timed(seeded, args.steps)
    # the floor of e2e: this step's offset bytes over PCIe with nothing else going on (all ranks copy at the same time,
    # like in the step; on a piece of at most 2 GiB), from the same host buffer
    up_bytes = int(stats_e2e[-1]["upload_bytes"])
    piece = min(up_bytes, 2 << 30)
    src_u8 = off_host.view(torch.uint8).reshape(-1)[:piece]
    dst_u8 = torch.empty(piece, dtype=torch.uint8, device="cuda")
    dst_u8.copy_(src_u8, non_blocking=True)
    ms_copy, _ = timed(lambda: dst_u8.copy_(src_u8, non_blocking=True), 2)
    h2d_alone = {"GBps_per_rank": piece / (ms_copy * 1e-3) / 1e9, "ms_for_this_step's_bytes": ms_copy * up_bytes / max(piece, 1),
                 "pinned": bool(off_host.is_pinned()),
                 "note": "cudaMemcpyAsync of the step's offset slice alone, all ranks at once: no schedule can bring e2e below this"}
    del dst_u8
    clocks = sampler.stop() if rank == 0 else None
    rays = total_rays(stats[-1])
    if args.dump_outputs:
        by_class = torch.tensor([float(stats[-1][k]) for k in RAY_CLASSES], dtype=torch.float64, device="cuda")
        if G > 1:
            dist.all_reduce(by_class, op=dist.ReduceOp.SUM)
    culled = torch.tensor([float(stats[-1]["rays_shadow_culled"])], dtype=torch.float64, device="cuda")
    if G > 1:
        dist.all_reduce(culled, op=dist.ReduceOp.SUM)
    culled_all = culled.item()   # (hit, light) pairs the reference queries and this path settles by l.n <= 0 alone
    value = rays / (ms_dev * 1e-3) / 1e6
    e2e_value = rays / (ms_e2e * 1e-3) / 1e6

    # per-rank kernel time of one frame (per-launch CUDA events on the library's stream, RH_FLAG_PROFILE): rank skew
    prof = [step_device(profile=True) for _ in range(2)][-1]
    per_rank = torch.tensor([prof["ms_trace"], prof["ms_shadow"], prof["ms_resolve"], prof["ms_total"]], dtype=torch.float64, device="cuda")
    all_ranks = [torch.zeros_like(per_rank) for _ in range(G)]
    if G > 1:
        dist.all_gather(all_ranks, per_rank)
    else:
        all_ranks = [per_rank]
    per_rank_ms = [{"trace": float(x[0]), "shadow": float(x[1]), "resolve": float(x[2]), "render_call_device": float(x[3])} for x in all_ranks]

    # roofline of the dominant kernel: per-launch times from those events, algorithmic bytes from the instrumented
    # kernels (RH_FLAG_COUNT), both live here; DRAM / L2 traffic and issue statistics from the committed ncu launch list
    cnt = step_device(count=True)
    ab = algorithmic_bytes(cnt, 0 if c5 else 16, bool(sc.tables_in_smem), rows * W, spp)
    peaks, peak_kind = load_peaks()
    shadow_refill = bool(prof.get("shadow_split"))
    walk_kernel = "shadow_refill_kernel" if shadow_refill else "shadow_pooled_kernel"
    kernels_ms = {"trace_kernel": prof["ms_trace"], "classify_kernel+" + walk_kernel: prof["ms_shadow"], "resolve_kernel": prof["ms_resolve"]}
    kernels_launches = {"trace_kernel": prof["trace_launches"], "classify_kernel+" + walk_kernel: prof["shadow_launches"], "resolve_kernel": 1}
    rb = sc.record_bytes
    record_set = {"trace_kernel": rb["nodes"] + rb["tris"] + rb["shade"] + rb["texels"], "classify_kernel+" + walk_kernel: rb["nodes"] + rb["tris"],
                  "resolve_kernel": 0}
    parts = {"trace_kernel": [ab["trace"]], "classify_kernel+" + walk_kernel: [ab["classify"], ab["walk"]], "resolve_kernel": [ab["resolve"]]}
    kernels_stream = {k: sum(x["stream"] for x in v) for k, v in parts.items()}
    kernels_gather = {k: sum(x["gather"] for x in v) for k, v in parts.items()}
    # of the gathers only one pass over the record set per launch has to come from HBM (classify + walk: the walk launches)
    walk_launches = {k: (n // 2 if "+" in k else n) for k, n in kernels_launches.items()}
    kernels_bytes = {k: kernels_stream[k] + min(kernels_gather[k], max(1, walk_launches[k]) * record_set[k]) for k in kernels_ms}
    dom = max(kernels_ms, key=kernels_ms.get)
    dom_ms, dom_bytes, dom_n = kernels_ms[dom], kernels_bytes[dom], max(1, kernels_launches[dom])
    achieved = dom_bytes / (dom_ms * 1e-3) / 1e9
    gather_l2, gather_hbm, stream_l2 = capi.C.c_double(), capi.C.c_double(), capi.C.c_double()
    capi.check(L.rh_bench_gather(4 << 20, 20, capi.C.byref(gather_l2)))
    capi.check(L.rh_bench_gather(4 << 30, 5, capi.C.byref(gather_hbm)))
    capi.check(L.rh_bench_stream(64 << 20, 20, capi.C.byref(stream_l2)))
    measured = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f).get(name)
        if tj and G == 1:
            ks = [k for k in dom.split("+") if k in tj["kernels"]]
            if ks:
                dram = sum(tj["kernels"][k]["dram_bytes_per_frame"] for k in ks)
                l2 = sum(tj["kernels"][k]["l2_bytes_per_frame"] for k in ks)
                ns = sum(tj["kernels"][k]["ms_per_frame_under_ncu"] for k in ks)
                inst = sum(tj["kernels"][k]["warp_instructions_per_frame"] for k in ks)
                measured = {"source": "profiles/" + tj["source"] + " (ncu launch list of one frame of this workload, same kernels)",
                            "dram_bytes_per_frame": dram, "l2_bytes_per_frame": l2, "ms_per_frame_under_ncu": ns,
                            "dram_frac": dram / (ns * 1e-3) / 1e9 / peaks["hbm_gbs"],
                            "l2_GBps": l2 / (ns * 1e-3) / 1e9, "l2_frac": l2 / (ns * 1e-3) / 1e9 / max(stream_l2.value, 1e-9),
                            "issue_active_pct": sum(tj["kernels"][k]["issue_active_pct"] * tj["kernels"][k]["ms_per_frame_under_ncu"] for k in ks) / ns,
                            "warps_active_pct": sum(tj["kernels"][k]["warps_active_pct"] * tj["kernels"][k]["ms_per_frame_under_ncu"] for k in ks) / ns,
                            "threads_per_inst": sum(tj["kernels"][k]["thread_instructions_per_frame"] for k in ks) / max(inst, 1)}
    except Exception:
        measured = None
    all_bytes = sum(kernels_bytes.values())
    roofline = {"bound": "issue", "memory_roofline": "hbm", "kernel": dom, "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": achieved / peaks["hbm_gbs"], "peak_kind": f"MEASURED_PEAKS.json hbm_gbs ({peak_kind})",
                "traffic": (measured["dram_bytes_per_frame"] / dom_n) if measured else None,
                "algorithmic_bytes_per_launch": dom_bytes / dom_n, "algorithmic_bytes_per_frame": dom_bytes,
                "kernel_ms_per_frame": dom_ms, "launches_per_frame": dom_n, "avg_launch_ms": dom_ms / dom_n,
                "kernel_share_of_frame": dom_ms / max(prof["ms_total"], 1e-9),
                "measured_under_ncu": measured,
                "all_kernels": {k: {"ms_per_frame": kernels_ms[k], "algorithmic_GB_per_frame": kernels_bytes[k] / 1e9,
                                    "GBps": kernels_bytes[k] / max(kernels_ms[k], 1e-9) / 1e6,
                                    "stream_GB_per_frame": kernels_stream[k] / 1e9, "gather_requests_GB_per_frame": kernels_gather[k] / 1e9,
                                    "gather_request_GBps": kernels_gather[k] / max(kernels_ms[k], 1e-9) / 1e6,
                                    "record_set_GB": record_set[k] / 1e9} for k in kernels_ms},
                "frame_check": {"algorithmic_GB_per_frame": all_bytes / 1e9, "GBps_over_the_step": all_bytes / (ms_dev * 1e-3) / 1e9,
                                "below_peak": bool(all_bytes / (ms_dev * 1e-3) / 1e9 <= peaks["hbm_gbs"])},
                "l2_stream_peak_GBps": stream_l2.value, "gather_peak_l2_resident_GBps": gather_l2.value,
                "gather_peak_hbm_resident_GBps": gather_hbm.value,
                "gather_request_frac_of_l2_gather_peak": kernels_gather[dom] / max(dom_ms, 1e-9) / 1e6 / max(gather_l2.value, 1e-9),
                "note": "algorithmic bytes = what has to cross HBM: the streams (offsets, queue entries written and read, accumulator "
                        "updates) + of the record gathers (nodes beyond the shared-memory-staged top levels, triangle / shading records, "
                        "texels; counted once per warp instruction) at most one pass over the record set per launch; the gather requests "
                        "themselves are served by L1 / L2 and are reported beside it (gather_request_GBps, against the measured random-gather "
                        "rate of an L2-resident set).  " + (
                            "The kernels are bound by instruction issue and dependent fp64 latency, not by memory — `frac` says how far below "
                            "the HBM roofline that leaves them" if not c5 else
                            "With 2.1 GB of records the walks are bound by the L1 / L2 gather path and by lane utilisation, not by HBM streaming")}

    # N > 1: the assembled frame must be the frame one GPU renders alone (SURVEY 8e parity gate); checked on rank 0
    # outside the timed region.  (c5 at full size: the 16 parity rows instead — one GPU alone needs ~20 s per frame.)
    assembled_ok = None
    if G > 1:
        step_device_nccl()
        step_device_fused()
        torch.cuda.synchronize()
        if rank == 0 and not c5:
            solo = torch.empty((H, W, 3), dtype=torch.uint8, device="cuda")
            rh.render_device(job, solo, spp=spp, **dev_kw)
            assembled_ok = bool(torch.equal(solo, full_dev)) and bool(torch.equal(solo, peers.frame))
            del solo
        elif rank == 0:
            assembled_ok = bool(torch.equal(full_dev, peers.frame))
    frame_dev = rgb_dev if G == 1 else peers.frame   # the complete frame, on this rank

    cpu, parity = None, None
    if rank == 0 and not args.no_cpu_baseline:
        if not c5:
            v, sample, ref, prows = c4_oracle_sample(sc, W, H, spp, off_host.numpy(), 15.0, want_ids=True)
            cpu = {"value": v, "unit": "Mrays/s", "cores": os.cpu_count() or 1, "kind": "port", "sample": sample}
            # parity of the frame the timed steps rendered, on every row the oracle just rendered: bytes and hit ids.
            # (No collective in here: only rank 0 runs this block.  At N > 1 the complete frame is in this rank's peer
            # frame since the assembled-frame check above.)
            if G == 1:
                step_device()
            torch.cuda.synchronize()
            gpu_rows = frame_dev[torch.from_numpy(prows).cuda()].cpu().numpy()
            ids_dev = torch.empty((H * W * spp, 2), dtype=torch.int32, device="cuda")
            rh.render_device(job, torch.empty((H, W, 3), dtype=torch.uint8, device="cuda"), spp=spp, hit_ids_dev=ids_dev, **dev_kw)
            gpu_ids = ids_dev.view(H, W, spp, 2)[torch.from_numpy(prows).cuda()].cpu().numpy()
            del ids_dev
            parity = compare_u8(gpu_rows, ref["rgb_u8"][prows])
            mism = np.any(gpu_ids != ref["hit_ids"][prows], axis=-1)
            parity.update(rows=int(len(prows)), of_rows=H, samples=int(mism.size), id_mismatches=int(mism.sum()),
                          against="oracle/oracle.cpp on the same offsets (parity unpinned by reference vectors: none exist, GHC absent)")
        else:
            prow, pcol = c5_sample_grid(W, H)
            v, sample, ref = c5_oracle_sample(sc, W, H, spp, seed, prow, pcol)
            cpu = {"value": v, "unit": "Mrays/s", "cores": os.cpu_count() or 1, "kind": "port", "sample": sample}
            # the 16 sample rows rendered once more as one "shard" of single-row bands (band r0 + k * (H / 16)), with hit ids
            r0, rstep = prow[0], prow[2]
            n_par = len(ref["rows"])
            rgb16 = torch.empty((L.rh_shard_rows(H, rstep, 1), W, 3), dtype=torch.uint8, device="cuda")
            ids16 = torch.empty((rgb16.shape[0] * W * spp, 2), dtype=torch.int32, device="cuda")
            rh.render_device(job, rgb16, spp=spp, seed=seed, shard_index=r0, shard_count=rstep, band_height=1, hit_ids_dev=ids16)
            torch.cuda.synchronize()
            ridx = torch.from_numpy(ref["rows"]).cuda()
            rows_equal = bool(torch.equal(rgb16[:n_par], frame_dev[ridx]))
            cidx = torch.from_numpy(ref["cols"]).cuda()
            gpu_px = frame_dev[ridx][:, cidx].cpu().numpy()
            gpu_ids = ids16.view(rgb16.shape[0], W, spp, 2)[:n_par][:, cidx].cpu().numpy()
            parity = compare_u8(gpu_px, ref["rgb_u8"])
            mism = np.any(gpu_ids != ref["hit_ids"], axis=-1)
            parity.update(rows=int(n_par), columns=int(len(ref["cols"])), samples=int(mism.size), id_mismatches=int(mism.sum()),
                          sample_rows_equal_the_timed_frame=rows_equal,
                          against="oracle/oracle.cpp on the same offsets (parity unpinned by reference vectors: none exist, GHC absent)")

    if rank == 0:
        st = stats[-1]
        e2e_note = ("limited by the H2D copy of the f64 offset slices (16 B per pixel sample per frame; every rank uploads its rows and the "
                    "ranks share the host's PCIe complex): see e2e_device_generated_offsets / `value` for the same frame without the upload")
        line = {"metric": wl["metric"], "value": value, "unit": "Mrays/s", "n_gpus": G, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
                "data": wl["data"], "config": config_dict(wl, G, name), "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": "Mrays/s", "ms_per_step": ms_e2e,
                        "h2d_bytes_per_step": int(stats_e2e[-1]["upload_bytes"]), "d2h_bytes_per_step": int((H if G > 1 else rows) * W * 3),
                        "h2d_alone": h2d_alone, "note": e2e_note},
                "gpu_launches": int(launches) * args.steps, "gpu_launches_per_step": int(launches),
                "rays_per_frame": rays, "frame_ms": ms_dev,
                "rays_by_class_rank0": {k: int(st[k]) for k in ("rays_primary", "rays_reflect", "rays_probe", "rays_exit", "rays_shadow",
                                                                "rays_shadow_culled", "shadow_walk_pairs")},
                "shadow_rays_note": "rays_shadow counts every shadowIntersection call of the reference (hits x lights); of those, "
                                    "rays_shadow_culled have l.n <= 0 (Lambert term exactly 0, no query needed) and shadow_walk_pairs "
                                    "had to walk a tree; the rest are settled by plane / sphere / root-box / light-map tests",
                "value_without_culled_shadow_pairs": (rays - culled_all) / (ms_dev * 1e-3) / 1e6,
                "shadow_walk_schedule": "per-lane refill" if shadow_refill else "pooled",
                "per_rank_kernel_ms": per_rank_ms, "setup": setup, "cold_start": cold,
                "roofline": roofline, "cpu_baseline": cpu, "parity": parity}
        if ms_seeded is not None:
            line["e2e_device_generated_offsets"] = {"value": rays / (ms_seeded * 1e-3) / 1e6, "unit": "Mrays/s", "ms_per_step": ms_seeded,
                                                    "h2d_bytes_per_step": 8, "d2h_bytes_per_step": int(rows * W * 3),
                                                    "note": "RH_OFFSETS_SPLITMIX64: same stream, same image, regenerated in the kernel; "
                                                            "informational — `e2e` above uploads the stream as north_star asks"}
        if assembled_ok is not None:
            line["assembled_frame_equals_single_gpu_frame" if not c5 else "both_exchanges_assemble_the_same_frame"] = assembled_ok
            line["exchange"] = exchange
        if dumped is not None:
            dump_outputs(args.dump_outputs, dumped, dump_idx, by_class.cpu().numpy())
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if G > 1:
        peers.close()
        dist.destroy_process_group()
    rh.shutdown()


if __name__ == "__main__":
    main()
