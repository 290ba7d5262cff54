#!/bin/bash
# Interleaved A/B of the headline bench between a reference build of the native library and the tree's build, plus the output
# comparison of both on the same seed.
# usage: tools/ab_native.sh <reference libqueasars_b200.so> <output directory> [rounds=3]
ref_lib=$(readlink -f "$1")
out=${2:?output directory}
rounds=${3:-3}
mkdir -p "$out"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$out/gpu.csv"
for i in $(seq 1 "$rounds"); do
  QB_NATIVE_LIB=$ref_lib timeout 600 python bench.py --steps 200 --skip-extras > "$out/ref_$i.json" 2> "$out/ref_$i.err"
  timeout 600 python bench.py --steps 200 --skip-extras > "$out/new_$i.json" 2> "$out/new_$i.err"
done
QB_NATIVE_LIB=$ref_lib timeout 600 python bench.py --steps 5 --skip-extras --dump-outputs "$out/dump_ref" > /dev/null 2>&1
timeout 600 python bench.py --steps 5 --skip-extras --dump-outputs "$out/dump_new" > /dev/null 2>&1
python - "$out" "$rounds" <<'PY'
import json, sys
import numpy as np
out, rounds = sys.argv[1], int(sys.argv[2])
print(open(f"{out}/gpu.csv").read().strip())
for arm in ("ref", "new"):
    vals = []
    for i in range(1, rounds + 1):
        try:
            d = json.loads(open(f"{out}/{arm}_{i}.json").read().strip().splitlines()[-1])
        except Exception as e:  # noqa: BLE001
            print(arm, i, "no result:", e)
            continue
        vals.append(d["value"])
        print(arm, i, "value", round(d["value"]), "e2e", round(d["e2e"]["value"]), "fp64 frac", round(d["roofline"]["fp64"]["frac"], 3), "clocks", d.get("clocks"))
    if vals:
        print(arm, "median", float(np.median(vals)), "range", min(vals), max(vals))
for name in ("values", "e2e_values"):
    a, b = np.load(f"{out}/dump_ref/{name}.npy"), np.load(f"{out}/dump_new/{name}.npy")
    print(name, a.shape, "max rel diff", float(np.max(np.abs(a - b) / np.maximum(1.0, np.abs(a)))))
PY
