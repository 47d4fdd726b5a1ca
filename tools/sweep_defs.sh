#!/bin/bash
# Rebuilds the traversal and shading kernels (kernels_trace.cu, kernels_shade.cu) with each set of compile-time knobs
# (make TRACE_DEFS=...) and runs a short bench for each.
# usage: tools/sweep_defs.sh "<defs 1>" "<defs 2>" ...   e.g. "" "-DRTC_TRACE_MIN_BLOCKS=6 -DRTC_FETCH_THRESHOLD=16"
# BENCH_ARGS overrides the bench flags (default: 4 steps of 32 spp).
BENCH_ARGS=${BENCH_ARGS:---steps 4 --warmup 3 --spp-per-step 32 --no-cpu-baseline --no-ncu --no-probes}
for cfg in "$@"; do
  touch tweeker_raytracer_b200/csrc/kernels_trace.cu tweeker_raytracer_b200/csrc/kernels_shade.cu
  make -s -j4 core host TRACE_DEFS="$cfg" > /tmp/sweep_build.log 2>&1 || { echo "build failed for $cfg"; tail -5 /tmp/sweep_build.log; continue; }
  echo "== $cfg"
  python bench.py $BENCH_ARGS 2>/tmp/sweep_err.log | tail -1 | python -c '
import sys, json
try:
    d = json.loads(sys.stdin.read()); r = d["roofline"]
    print(round(d["value"], 1), "Msamples/s", round(d["mrays_per_s"], 1), "Mrays/s; extend", round(r["extend_mrays_per_s"], 1), "connect", round(r["connect"]["mrays_per_s"], 1), "e2e", round(d["e2e"]["value"], 1), {k: round(v, 2) for k, v in r["per_ray"].items()}, {k: round(v, 3) for k, v in r["kernel_share_of_step"].items()}, "ms/step", round(d["ms_per_step"], 2))
except Exception as e:
    print("bench failed:", e)' || tail -5 /tmp/sweep_err.log
done
