#!/bin/bash
# One-GPU evidence of the tangent-form change: build, -m gpu suite, smoke, interleaved A/B against the parent's library
# (built into queasars_b200/csrc/variants/lib_parent.so beforehand), one full bench of each build.
# usage: tools/gpu_tangent_round.sh <output directory>
out=${1:?output directory}
mkdir -p "$out"
python -c "import __graft_entry__ as g; g.build()" > "$out/t_build.log" 2>&1; echo "build rc=$?"
timeout 1200 python -m pytest tests -m gpu -q > "$out/t_tests.log" 2>&1; echo "pytest rc=$?"; tail -n 5 "$out/t_tests.log"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > "$out/t_smoke.log" 2>&1; echo "smoke rc=$?"; tail -n 2 "$out/t_smoke.log"
bash tools/ab_native.sh queasars_b200/csrc/variants/lib_parent.so "$out/ab" 3
timeout 1500 python bench.py > "$out/t_bench_full.json" 2> "$out/t_bench_full.err"; echo "full bench rc=$?"
QB_NATIVE_LIB=$(readlink -f queasars_b200/csrc/variants/lib_parent.so) timeout 1500 python bench.py > "$out/t_bench_full_ref.json" 2> "$out/t_bench_full_ref.err"
echo "full bench (parent) rc=$?"
python - "$out" <<'PY'
import json, sys
out = sys.argv[1]
for arm in ("t_bench_full", "t_bench_full_ref"):
    try:
        d = json.loads(open(f"{out}/{arm}.json").read().strip().splitlines()[-1])
    except Exception as e:  # noqa: BLE001
        print(arm, "no result:", e)
        continue
    print("==", arm, "value", d["value"], "e2e", d["e2e"]["value"], "fp64 frac", d["roofline"]["fp64"]["frac"], "clocks", d.get("clocks"))
    for k in ("optimizer_calls", "c3_24q_tfim", "c4_26q_sampler", "c2_complex64"):
        print(k, json.dumps(d.get(k))[:400])
    for n, v in d.get("gate_apply", {}).items():
        print(n, json.dumps(v)[:300])
PY
