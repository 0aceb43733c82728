#!/bin/bash
# C4 under torchrun on N GPUs: band heights (rows per interleaved band).  Short runs
# (no CPU baseline, no cold start); one JSON line per configuration into gpurun_out/.
N=${N:-8}
mkdir -p gpurun_out
run() {  # tag, env, extra args
  env $2 timeout 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29511 \
    bench.py --gpus $N --workload c4 --no-cpu-baseline --no-cold-start $3 > gpurun_out/ab_${N}gpu_$1.json 2> gpurun_out/ab_${N}gpu_$1.err
  python - <<PY
import json
try:
    d = json.loads(open("gpurun_out/ab_${N}gpu_$1.json").read().strip().splitlines()[-1])
    pr = d["per_rank_kernel_ms"]
    print("$1", "ms %.3f" % d["ms_per_step"], "e2e %.2f" % d["e2e"]["ms_per_step"], "assembled", d.get("assembled_frame_equals_single_gpu_frame"),
          "rank call ms min %.2f max %.2f" % (min(x["render_call_device"] for x in pr), max(x["render_call_device"] for x in pr)))
except Exception as e:
    print("$1 no line:", e)
PY
}
run bh16 "" "--band-height 16"
run bh4 "" "--band-height 4"
run bh1 "" "--band-height 1"
