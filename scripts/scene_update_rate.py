"""Cost of scene updates (rh_scene_update) against rebuilding the scene (rh_scene_create), on the bench view of
dragon_full and on the synthetic configs[4] scene (rh_make_synthetic: 10 M triangles + 1 000 spheres, 3 point lights).

    python scripts/scene_update_rate.py [--scenes dragon_full,c5] [--reps 5] [--width 3840 --height 2160] [--json out.json]

Per scene: rh_scene_create of the flattened description (the flattening itself is not timed), then updates of each
kind, alternating an edit and its inverse so that every timed call changes bytes: colours only (every material's
color1), one point light moved, every light moved, and one mesh's material toggled to Emmit and back.  Every call is
timed with the host clock around the call, which returns after the device work; reported are the minimum and median
of the 2 x --reps calls, of the edits and of the reverts, and the rh_update_info of the last call.  Then the interactive loop: move a light, reset an
accumulator and make one 1-spp rh_render_accumulate call at --width x --height (SplitMix64 seed 24), --reps times;
reported are the update, the call and the sum.  The card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import rayhs_b200 as rh  # noqa: E402
from rayhs_b200 import capi  # noqa: E402
from ray_query_rate import card  # noqa: E402


def ms(f) -> tuple[float, object]:
    t = time.perf_counter()
    r = f()
    return (time.perf_counter() - t) * 1e3, r


def summary(xs):
    return {"min_ms": round(min(xs), 3), "median_ms": round(statistics.median(xs), 3), "n": len(xs)}


def mesh_material(sc):
    raw = sc.raw.contents
    for i in range(raw.n_objects):
        if raw.objects[i].kind == capi.RH_OBJ_MESH:
            return raw.objects[i].material
    return None


def measure(sc, reps: int, width: int, height: int) -> dict:
    L = capi.lib()
    flat = sc.flat
    creates = []
    for _ in range(max(2, reps // 2)):
        h = C.c_void_p()
        t, _ = ms(lambda: capi.check(L.rh_scene_create(flat, C.byref(h))))
        creates.append(t)
        ms3 = (C.c_double * 3)()
        L.rh_scene_info(h, ms3, None)
        L.rh_scene_destroy(h)
    out = {"create": summary(creates), "create_stages_ms": {"trees": ms3[0], "light_tables": ms3[1], "upload": ms3[2]}}
    sc.device
    base_m, base_l = sc.materials, list(sc.lights)
    points = [i for i, x in enumerate(base_l) if x.kind == capi.RH_LIGHT_POINT]
    mm = mesh_material(sc)

    def colours(k):
        m = sc.materials
        for x in m:
            x.color1[:] = [c * (0.9 if k % 2 == 0 else 1 / 0.9) for c in x.color1]
        return dict(materials=m)

    def move(which):
        def f(k):
            l = list(sc.lights)
            for i in which:
                l[i].vec[1] += 0.05 if k % 2 == 0 else -0.05
            return dict(lights=l)
        return f

    def emmit(k):
        m = sc.materials
        m[mm].kind = capi.RH_MAT_EMMIT if k % 2 == 0 else base_m[mm].kind
        return dict(materials=m)

    kinds = {"colours_only": colours, "one_point_light": move(points[:1]), "all_lights": move(range(len(base_l)))}
    if mm is not None:
        kinds["emitter_toggle"] = emmit
    for name, edit in kinds.items():
        times, info = [], None
        for k in range(2 * reps):
            args = edit(k)
            t, info = ms(lambda: sc.update(**args))
            times.append(t)
        # (an emitter toggle differs by direction: with the mesh an emitter the scene may have no light tables at all)
        out[name] = dict(summary(times), edit=summary(times[0::2]), revert=summary(times[1::2]), info=info)
    sc.update(materials=base_m, lights=base_l)
    # interactive loop: move a light, one 1-spp progressive call
    job = rh.renderingFromScene(sc, width, height)
    acc = rh.Accumulator(job, stream_spp=1, device=True)
    acc.add(1, seed=24, linear=False)  # warm-up of the frame's buffers
    move_one = move(points[:1] if points else [0])
    ups, calls, device = [], [], []
    for k in range(reps):
        args = move_one(k)
        t_up, _ = ms(lambda: sc.update(**args))
        acc.reset()
        t_call, img = ms(lambda: acc.add(1, seed=24, linear=False))
        import torch

        torch.cuda.synchronize()
        ups.append(t_up)
        calls.append(t_call)
        device.append(img.stats["ms_total"])
    acc.close()
    out["interactive_loop"] = {"width": width, "height": height, "update": summary(ups), "accumulate_1spp": summary(calls),
                               "accumulate_ms_total": summary(device), "sum": summary([a + b for a, b in zip(ups, calls)])}
    return out


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--scenes", default="dragon_full,c5")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--json", default=None, help="also write the result here")
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("scene_update_rate.py measures on the GPU; no CUDA device here")
    rh.init()
    res = {"card": card()}
    for name in a.scenes.split(","):
        if name == "c5":
            sc = rh.Scene.synthetic(10_000_000, 1000)
        else:
            sc = rh.Scene.from_pack(os.path.join(ROOT, "tests", "golden", name + ".pack"))
        t, _ = ms(lambda: sc.flat)
        r = measure(sc, a.reps, a.width, a.height)
        r["flatten_ms"] = round(t, 1)
        res[name] = r
        print(name, json.dumps(r), flush=True)
        sc.close()
    print(json.dumps(res["card"]))
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)
    return 0


if __name__ == "__main__":
    sys.exit(main())
