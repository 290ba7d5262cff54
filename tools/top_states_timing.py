"""Most probable basis states on the device (qb_top_states, and the sharded select on one GPU): passes, time per select pass and
bytes per pass against a read ceiling measured in the same run, the collect and the sort, the end-to-end call, and for comparison
the circuit itself and 10 000 shots of the same states.

Kernel times are GPU timestamps of torch.profiler (CUDA activities) summed per kernel family over the timed calls, in a profiled
pass of their own; end-to-end times are host clocks around calls that end in a device synchronise, profiler off.  A select pass
is one top_select_kernel launch (all states of the batch together), so passes = select launches per call.  Bytes per pass = the
states it reads (batch x 2^n x 16 B); the read ceiling is a float64 torch.sum over a 4 GiB buffer (well above the L2).

    python tools/top_states_timing.py --out profiles/top_states_timing_b200.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
from oracle import evqe_genome as og  # noqa: E402
from queasars_b200 import gate_list as gl  # noqa: E402
from queasars_b200.engine import Engine  # noqa: E402
from tests.test_frontend_planner import build_circuit  # noqa: E402

FAMILIES = {"top_select_kernel": "select", "top_collect_kernel": "collect", "DeviceRadixSort": "sort", "sweep_kernel": "circuit",
            "bind_kernel": "circuit"}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def read_ceiling_gbs(reps=20):
    import torch

    x = torch.ones(1 << 29, dtype=torch.float64, device="cuda")  # 4 GiB
    for _ in range(3):
        x.sum()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        x.sum()
    end.record()
    torch.cuda.synchronize()
    ms = start.elapsed_time(end) / reps
    del x
    torch.cuda.empty_cache()
    return (8 << 29) / (ms * 1e-3) / 1e9


def kernels(fn, reps):
    """GPU ms per call by family, and launches per call by family."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    ms, launches = {}, {}
    for evt in prof.key_averages():
        fam = next((f for key, f in FAMILIES.items() if key in evt.key), None)
        if fam is None:
            continue
        total = getattr(evt, "device_time_total", None) or getattr(evt, "cuda_time_total", 0.0)
        ms[fam] = ms.get(fam, 0.0) + total / 1e3 / reps
        launches[fam] = launches.get(fam, 0) + evt.count / reps
    return ms, launches


def wall_ms(fn, reps):
    fn()
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        times.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(times))


def population(engine, n, count, seed):
    plans, values = [], []
    for s in range(count):
        genome, vals = og.random_individual(n, 6, True, seed + s)
        plans.append(engine.compile(gl.from_circuit(build_circuit(og.individual_circuit(genome, vals), n)), drop_final_phases=True))
        values.append(list(vals))
    return plans, values


def one_gpu_case(engine, n, batch, max_states, ceiling, reps):
    plans, values = population(engine, n, batch, 1000 + n)
    top = lambda: engine.top_states(plans, values, max_states)  # noqa: E731
    top()
    ms, launches = kernels(top, reps)
    passes = launches.get("select", 0.0)
    per_pass = ms.get("select", 0.0) / max(passes, 1)
    pass_bytes = batch * (16 << n)
    rng = np.random.default_rng(0)
    uniforms = rng.random((batch, 10_000))
    return {
        "qubits": n, "batch": batch, "max_states": max_states, "passes": passes, "select_ms_per_pass": per_pass,
        "bytes_per_pass": pass_bytes, "select_gb_s": pass_bytes / (per_pass * 1e-3) / 1e9 if per_pass else None,
        "select_share_of_read_ceiling": (pass_bytes / (per_pass * 1e-3) / 1e9) / ceiling if per_pass else None,
        "collect_ms": ms.get("collect", 0.0), "collect_launches": launches.get("collect", 0.0), "sort_ms": ms.get("sort", 0.0),
        "circuit_kernels_ms": ms.get("circuit", 0.0), "top_states_call_ms": wall_ms(top, reps),
        "sample_10000_shots_call_ms": wall_ms(lambda: engine.sample(plans, values, 10_000, uniforms), reps),
        "entries_found": [int(idx.size) for idx, _ in top()[:2]],
    }


def sharded_case(engine, n, shards, max_states, reps):
    from queasars_b200.sharded import LocalShardedStatevector

    genome, vals = og.random_individual(n, 6, True, 2000 + n)
    gates = gl.from_circuit(build_circuit(og.individual_circuit(genome, vals), n))
    sv = LocalShardedStatevector(n, [engine] * shards, min_local=8)
    try:
        sv.run(gates, vals)
        ms = wall_ms(lambda: sv.top_states(max_states), reps)
        return {"qubits": n, "shards_on_one_gpu": shards, "max_states": max_states, "passes": sv.top_passes, "top_states_call_ms": ms,
                "swaps_done": sv.swaps_done}
    finally:
        sv.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--quick", action="store_true", help="small sizes only (a rehearsal)")
    args = ap.parse_args()
    result = {"card": card(), "method": __doc__.strip().splitlines()[0]}
    result["read_ceiling_gb_s"] = ceiling = read_ceiling_gbs()
    engine = Engine(device=0, dtype="complex128")
    sizes = ((14, 4), (16, 2)) if args.quick else ((20, 32), (26, 4), (30, 1))
    result["one_gpu"] = [one_gpu_case(engine, n, batch, m, ceiling, args.reps) for n, batch in sizes for m in (1, 1024, 1 << 20)]
    n_sharded = 16 if args.quick else 30
    result["sharded"] = [sharded_case(engine, n_sharded, 2, m, args.reps) for m in (1, 1024, 1 << 20)]
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
