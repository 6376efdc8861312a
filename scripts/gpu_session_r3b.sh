#!/bin/bash
TAG=${1:-r3x}; OUT=gpurun_out; mkdir -p $OUT
timeout 1800 python -m pytest tests -m gpu -q -x --durations=5 > $OUT/${TAG}_pytest.log 2>&1; tail -9 $OUT/${TAG}_pytest.log | cut -c1-220
python scripts/time_vertex_grads.py 2>&1 | grep -v Warning | tail -3 | tee $OUT/${TAG}_vertex_grads.txt
( time python bench.py ) > $OUT/${TAG}_bench.json 2> $OUT/${TAG}_bench.err; tail -4 $OUT/${TAG}_bench.err
python - <<PY
import json
try:
    d = json.load(open("$OUT/${TAG}_bench.json"))
    def show(name, r):
        rf = r["roofline"]
        print(name, "value", r["value"], "ms", r["ms_per_step"], "med", r.get("ms_per_step_median"), "fwd", r["forward_only"]["ms_per_step"],
              "e2e", r["e2e"]["value"], r["e2e"]["ms_per_step"], "top", rf["kernel"], rf["kernel_ms"], "frac", rf["frac"], "step_frac", rf["step"]["frac"],
              "launches", r["gpu_launches"])
        print("   kernels", {k: v["ms_per_step"] for k, v in rf["kernels"].items()})
        if "parity" in r:
            p = r["parity"]; print("   parity", p["pass"], p["index_mismatches"], p["image_max_abs_err"], p["grad_camera_max_rel_err"], "| cpu", r["cpu_baseline"]["value"], r["cpu_baseline"]["sample"][:60])
    show("c2_mesh", d)
    for k, r in d.get("extra", {}).items():
        if "roofline" in r: show(k, r)
        else: print(k, r)
except Exception as e:
    print("bench FAILED", repr(e))
PY
