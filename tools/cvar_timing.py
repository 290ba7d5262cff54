"""Exact CVaR on the device (qb_evaluate_cvar): cost of the order-data build, of the sweeps and of the CVaR kernels
(cvar_chunk_kernel + two scans + cvar_finish_kernel), achieved bytes/s of the chunk kernel against its byte model, and the sampled
route (10 000 shots through B200OperatorSamplerCircuitEvaluator) end to end for comparison.

Kernel times are GPU timestamps of torch.profiler (CUDA activities, CUPTI) summed per kernel name over the timed calls, in a
profiled pass of their own (kernels that overlap on two streams are summed, not merged); end-to-end times are host clocks
around calls that end in a device synchronise, profiler off.  The order-data build time is the first call on a new Hamiltonian
minus a warm call, after a throwaway Hamiltonian of the same width has loaded the kernels.

    python tools/cvar_timing.py --out profiles/cvar_timing_b200.json
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
from queasars_b200 import B200OperatorSamplerCircuitEvaluator, B200SamplerV2  # noqa: E402
from queasars_b200 import gate_list as gl  # noqa: E402
from queasars_b200.engine import Engine  # noqa: E402
from queasars_b200.operators import SparsePauliOp  # noqa: E402
from tests.test_frontend_planner import build_circuit  # noqa: E402
from tests.test_gpu_parity import random_ising  # noqa: E402

CVAR_KERNELS = ("cvar_chunk_kernel", "scan_chunks_kernel", "cvar_finish_kernel")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def population(n, count, seed):
    out = []
    for s in range(count):
        genome, values = og.random_individual(n, 6, True, seed + s)
        out.append((build_circuit(og.individual_circuit(genome, values), n), list(values)))
    return out


def kernel_ms(fn, reps):
    """GPU time per call of every kernel `fn` launches, by kernel family."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for evt in prof.key_averages():
        total = getattr(evt, "device_time_total", None) or getattr(evt, "cuda_time_total", 0.0)
        for fam in ("sweep_kernel", "bind_kernel") + CVAR_KERNELS:
            if fam in evt.key:
                out[fam] = out.get(fam, 0.0) + total / 1e3 / reps  # us -> ms per call
    return out


def wall_ms(fn, reps):
    fn()
    best = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        best.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(best))


def case(engine, label, op, circuits, alpha, reps):
    n = op.num_qubits
    ham = engine.hamiltonian(op, build_table=False)
    plans = [engine.compile(gl.from_circuit(c), drop_final_phases=True) for c, _ in circuits]
    params = [v for _, v in circuits]
    # a throwaway Hamiltonian of the same width first: loads the CVaR / CUB kernel modules and sizes the engine's state buffers,
    # so the first call below pays the order-data build itself (kernels, and cudaMalloc / cudaFree of its buffers) and nothing else
    engine.cvar(plans[:1], params[:1], engine.hamiltonian(op, build_table=False), alpha)
    t0 = time.perf_counter()
    engine.cvar(plans[:1], params[:1], ham, alpha)  # builds the order data
    first_ms = (time.perf_counter() - t0) * 1e3
    one_ms = wall_ms(lambda: engine.cvar(plans[:1], params[:1], ham, alpha), reps)
    call_ms = wall_ms(lambda: engine.cvar(plans, params, ham, alpha), reps)
    ks = kernel_ms(lambda: engine.cvar(plans, params, ham, alpha), reps)
    cvar_ms = sum(ks.get(k, 0.0) for k in CVAR_KERNELS)
    n_eff = max(n, engine.tile_bits)
    amp = 16 if engine.dtype == "complex128" else 8
    model_bytes = len(plans) * (1 << n_eff) * (4 + 8 + amp)  # perm + E sorted + one gathered amplitude
    sector_bytes = len(plans) * (1 << n_eff) * (4 + 8 + 32)  # the gathered amplitude moves a whole 32 B sector
    chunk_ms = ks.get("cvar_chunk_kernel", float("nan"))
    return {
        "case": label, "n_qubits": n, "individuals": len(plans), "alpha": alpha, "dtype": engine.dtype,
        "order_build_ms": first_ms - one_ms, "first_call_ms": first_ms,
        "call_ms_end_to_end": call_ms,
        "kernel_ms_per_call": ks, "cvar_kernels_ms": cvar_ms, "cvar_share_of_call": cvar_ms / call_ms,
        # sweep_kernel durations summed: from 8 states on, the sweeps of two circuit groups run on two streams at once, and the sum
        # then exceeds the sweeps' share of the call's wall time
        "sweep_kernels_summed_ms": ks.get("sweep_kernel", 0.0), "sweep_streams": 2 if len(plans) >= 8 else 1,
        "chunk_kernel_model_bytes": model_bytes, "chunk_kernel_GBps_model": model_bytes / chunk_ms / 1e6,
        "chunk_kernel_GBps_sectors": sector_bytes / chunk_ms / 1e6,
    }


def sampled_route(op, circuits, alpha, reps):
    sampler = B200SamplerV2(device=0, seed=1)
    cs, vs = [c for c, _ in circuits], [v for _, v in circuits]
    shots = B200OperatorSamplerCircuitEvaluator(sampler, 10000, op, alpha)
    exact = B200OperatorSamplerCircuitEvaluator(sampler, None, op, alpha)
    return {"sampled_10000_shots_ms": wall_ms(lambda: shots.evaluate_circuits(cs, vs), reps),
            "exact_ms": wall_ms(lambda: exact.evaluate_circuits(cs, vs), reps)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    golden = json.load(open(os.path.join(ROOT, "tests", "golden", "jssp_hamiltonians.json")))
    entry = golden["jssp_26q"]
    jssp = SparsePauliOp._raw(26, [0] * len(entry["z_masks"]), entry["z_masks"], entry["coeffs"])
    ising = SparsePauliOp.from_list(random_ising(20))
    engine = Engine(device=0)
    pop20 = population(20, 32, 100)
    pop26 = population(26, 4, 200)
    result = {"card": card(), "method": __doc__.split("\n\n")[1].replace("\n", " "), "cases": []}
    result["cases"].append(case(engine, "20q x 32 random_ising", ising, pop20, 0.5, args.reps))
    result["cases"].append(case(engine, "26q JSSP x 1", jssp, pop26[:1], 0.5, args.reps))
    result["cases"].append(case(engine, "26q JSSP x 4", jssp, pop26, 0.5, args.reps))
    result["end_to_end_evaluator"] = {
        "20q x 32 random_ising": sampled_route(ising, pop20, 0.5, args.reps),
        "26q JSSP x 1": sampled_route(jssp, pop26[:1], 0.5, args.reps),
        "26q JSSP x 4": sampled_route(jssp, pop26, 0.5, args.reps),
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
