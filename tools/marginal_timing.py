"""Exact marginal probabilities on the device (qb_marginal_device, the kernel behind qb_marginal_probabilities): device time per
call at 26, 28 and 30 qubits (complex128) for m in {1, 8, 16, 24} measured qubits, low-bit (0..m-1) and high-bit (n-m..n-1)
subsets, and the bytes read over that time against the copy and read bandwidth of profiles/r2_hbm_directional.json and a read
ceiling measured in the same run.

The state is a random EVQE circuit's, applied once into a caller-owned device buffer, so the timed work is the marginal alone.
Kernel time = GPU timestamps of torch.profiler (CUDA activities) summed over marginal_kernel and marginal_reduce_kernel, per call,
in a profiled pass of its own; call time = CUDA events on the engine's stream around the whole call (kernels plus the copy of the
2^m doubles to pageable host memory), profiler off.  Bytes = the state read once (2^n x 16 B); the output (2^m x 8 B, plus partial
rows) is listed apart.  The state (1 GiB and more) is far above the 126 MB L2, so every call reads HBM.

    python tools/marginal_timing.py --out profiles/marginal_timing_b200.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
from oracle import evqe_genome as og  # noqa: E402
from queasars_b200 import gate_list as gl  # noqa: E402
from queasars_b200.engine import Engine  # noqa: E402
from tests.test_frontend_planner import build_circuit  # noqa: E402

FAMILIES = {"marginal_reduce_kernel": "reduce", "marginal_kernel": "marginal"}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def hbm_reference():
    with open(os.path.join(ROOT, "profiles", "r2_hbm_directional.json")) as fh:
        d = json.load(fh)
    return {"read_only_sum_gb_s": d["16GiB"]["read_only_sum"]["GBps"], "copy_gb_s": d["16GiB"]["copy"]["GBps"], "source": "profiles/r2_hbm_directional.json, 16 GiB"}


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


def kernel_ms(fn, reps):
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


def event_ms(engine, fn, reps):
    import torch

    stream = torch.cuda.ExternalStream(engine.stream) if engine.stream else torch.cuda.default_stream()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    start.record(stream)
    for _ in range(reps):
        fn()
    end.record(stream)
    end.synchronize()
    return start.elapsed_time(end) / reps


def state_case(engine, n, ms_list, ceiling, hbm, reps):
    genome, vals = og.random_individual(n, 4, True, 3000 + n)
    plan = engine.compile(gl.from_circuit(build_circuit(og.individual_circuit(genome, vals), n)), from_zero_state=False)
    ptr = engine.device_alloc(16 << n)
    rows = []
    try:
        engine.apply_plan_device(plan, vals, ptr, True)
        for m in ms_list:
            for kind, positions in (("low", list(range(m))), ("high", list(range(n - m, n)))):
                call = lambda: engine.marginal_device("complex128", n, ptr, 0, positions)  # noqa: E731
                total = float(call().sum())
                ms, launches = kernel_ms(call, reps)
                k_ms = ms.get("marginal", 0.0) + ms.get("reduce", 0.0)
                state_bytes = 16 << n
                gbs = state_bytes / (k_ms * 1e-3) / 1e9 if k_ms else None
                rows.append({
                    "qubits": n, "m": m, "subset": kind, "state_bytes": state_bytes, "output_bytes": 8 << m,
                    "kernel_ms": k_ms, "marginal_kernel_ms": ms.get("marginal", 0.0), "reduce_kernel_ms": ms.get("reduce", 0.0),
                    "launches_per_call": launches, "read_gb_s": gbs,
                    "share_of_read_ceiling_this_run": gbs / ceiling if gbs else None,
                    "share_of_r2_read_only_sum": gbs / hbm["read_only_sum_gb_s"] if gbs else None,
                    "share_of_r2_copy": gbs / hbm["copy_gb_s"] if gbs else None,
                    "call_ms_events": event_ms(engine, call, reps), "marginal_sum": total,
                })
                print(json.dumps(rows[-1]), flush=True)
    finally:
        engine.synchronize()
        engine.device_free(ptr)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--quick", action="store_true", help="small sizes only (a rehearsal)")
    args = ap.parse_args()
    result = {"card": card(), "method": __doc__.strip().splitlines()[0], "hbm_reference": hbm_reference()}
    result["read_ceiling_gb_s_this_run"] = ceiling = read_ceiling_gbs()
    engine = Engine(device=0, dtype="complex128")
    sizes = (16, 18) if args.quick else (26, 28, 30)
    ms_list = (1, 8, 12) if args.quick else (1, 8, 16, 24)
    result["cases"] = [row for n in sizes for row in state_case(engine, n, ms_list, ceiling, result["hbm_reference"], args.reps)]
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
