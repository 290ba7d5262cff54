"""Global <-> local exchange of a sharded statevector: the in-place kernel (swap_inplace_p2p_kernel, one buffer per shard, half
of the crossing bytes as peer loads) against the ping-pong kernel (swap_p2p_kernel, two buffers, peer stores only), alternated on
the same state in the same process, and a full EVQE-like run at a width only one buffer per GPU holds.

Swap times are host clocks around every shard's kernel launched through the engine API (``swap_global_inplace_p2p`` on the
shard buffers, ``swap_global_p2p`` from them into a second set), each ending in a device synchronise, joined over the shards;
median of `--reps` after one warm-up of each kernel; the two kernels alternate A B B A.  Bytes per GPU and direction:
(1 - 2^-g) 16 2^n_local, the same for both kernels.  A case "n:shards" puts every shard on a GPU of its own (NVLink) and is
recorded as not measured when the box has fewer GPUs; "n:shardsv" runs the shards round robin on the visible GPUs, several
virtual shards on one GPU exchanging through HBM, and the record says so.

    python tools/sharded_inplace_timing.py --out profiles/sharded_inplace_timing_b200.json
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
from oracle import evqe_genome as og  # noqa: E402
from queasars_b200 import _native  # noqa: E402
from queasars_b200 import gate_list as gl  # noqa: E402
from queasars_b200.primitives import get_engine  # noqa: E402
from tests.test_frontend_planner import build_circuit  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    rows = [[s.strip() for s in line.split(",")] for line in q.stdout.strip().splitlines()]
    return {"name": rows[0][0], "power_limit": rows[0][1], "gpus": len(rows), "power_limits": sorted({r[1] for r in rows})}


def free_bytes(devices):
    import torch

    return min(torch.cuda.mem_get_info(d)[0] for d in devices)


def swap_case(n, shards, virtual, reps):
    """Both exchange kernels through the engine API on raw shard buffers (one set for the in-place kernel, a second as the
    ping-pong kernel's destination).  ``virtual``: the shards go round robin over the visible GPUs (HBM, not NVLink); otherwise
    every shard needs a GPU of its own and the case is recorded as not measured on a smaller box."""
    from concurrent.futures import ThreadPoolExecutor

    n_dev = _native.device_count()
    g = int(math.log2(shards))
    nl = n - g
    shard_bytes = 16 << nl
    rec = {"n": n, "shards": shards, "n_local": nl, "shard_GiB": shard_bytes / 2**30}
    if not virtual and n_dev < shards:
        rec["status"] = f"not measured: one GPU per shard (NVLink) needs {shards} GPUs, {n_dev} visible"
        return rec
    per_gpu = -(-shards // n_dev) if virtual else 1
    devices = sorted({r % n_dev for r in range(shards)})
    rec.update(gpus=len(devices), link="NVLink (one shard per GPU)" if per_gpu == 1 else f"HBM ({per_gpu} virtual shards per GPU)")
    free = free_bytes(devices)
    if 2 * shard_bytes * per_gpu + (2 << 30) > free:
        rec["status"] = f"not measured: {2 * shard_bytes * per_gpu / 2**30:.0f} GiB of shard buffers per GPU, {free / 2**30:.0f} GiB free"
        return rec
    engines = [get_engine(r % n_dev) for r in range(shards)]
    for e in set(engines):
        for d in devices:
            e.enable_peer_access(d)
    lp = list(range(nl - g, nl))
    state, spare = [], []
    pool = ThreadPoolExecutor(max_workers=shards)
    try:
        for r, e in enumerate(engines):
            state.append(e.device_alloc(shard_bytes))
            spare.append(e.device_alloc(shard_bytes))

        def each(fn):  # every shard's kernel concurrently; returns when all of them completed (the after barrier)
            list(pool.map(fn, range(shards)))

        def inplace(r):
            engines[r].swap_global_inplace_p2p("complex128", nl, state, r, lp)
            engines[r].synchronize()

        def out_of_place(r):
            engines[r].swap_global_p2p("complex128", nl, state[r], spare, r, lp)
            engines[r].synchronize()

        kernels = {"inplace": inplace, "out_of_place": out_of_place}

        def timed(name):
            each(lambda r: engines[r].synchronize())  # the before barrier of the in-place kernel
            t0 = time.perf_counter()
            each(kernels[name])
            return time.perf_counter() - t0

        for name in kernels:
            timed(name)  # warm-up
        times = {name: [] for name in kernels}
        for rep in range(reps):
            for name in (list(kernels) if rep % 2 == 0 else list(kernels)[::-1]):
                times[name].append(timed(name))
    finally:
        pool.shutdown(wait=True)
        for e in set(engines):
            e.synchronize()
        for r, e in enumerate(engines):
            for ptr in (state[r:r + 1] + spare[r:r + 1]):
                e.device_free(ptr)
    cross = (1 - 2.0**-g) * shard_bytes
    rec["bytes_per_gpu_per_direction"] = cross * per_gpu
    for name, ts in times.items():
        t = float(np.median(ts))
        rec[f"{name}_s"], rec[f"{name}_all_s"] = t, ts
        rec[f"{name}_GBps_per_direction"] = cross * per_gpu / t / 1e9
    rec["inplace_over_out_of_place"] = rec["inplace_s"] / rec["out_of_place_s"]
    return rec


def evqe_run(n, shards, reps, shots):
    """Circuit, diagonal <H>, `shots` samples and uncached CVaR(0.5) on a state that only fits with one buffer per GPU."""
    from queasars_b200.sharded import LocalShardedStatevector

    n_dev = _native.device_count()
    if n_dev < shards:
        return {"n": n, "shards": shards, "status": f"not measured: {n_dev} GPU(s) visible"}
    engines = [get_engine(d) for d in range(shards)]
    sv = LocalShardedStatevector(n, engines)
    genome, values = og.random_individual(n, 4, True, 3600 + n)
    gates = gl.from_circuit(build_circuit(og.individual_circuit(genome, values), n))
    rng = np.random.default_rng(7)
    z = [1 << q for q in range(n)] + [(1 << q) | (1 << ((q + 1) % n)) for q in range(n)]
    c = [float(v) for v in rng.normal(size=len(z))]
    rec = {"n": n, "shards": shards, "buffers": sv.buffers, "circuit_ops": len(gates.ops), "shots": shots}

    def clock(fn):
        t0 = time.perf_counter()
        out = fn()
        for e in engines:
            e.synchronize()
        return time.perf_counter() - t0, out

    runs = []
    for _ in range(reps):
        sv.reset()
        before = sv.swaps_done
        t, _ = clock(lambda: sv.run(gates, values))
        runs.append((t, sv.swaps_done - before))
    rec["circuit_s"] = float(np.median([t for t, _ in runs]))
    rec["swaps_in_circuit"] = runs[-1][1]
    rec["expectation_s"], rec["expectation"] = clock(lambda: sv.diagonal_expectation(z, c))
    rec["norm"] = sv.norm_squared()
    uniforms = np.random.default_rng(1).random(shots)
    rec["sample_s"], _ = clock(lambda: sv.sample(shots, uniforms=uniforms))
    rec["cvar_0.5_uncached_s"], (value, stop) = clock(lambda: sv.cvar(z, c, 0.5, cache=False))
    rec["cvar_0.5"], rec["cvar_passes"] = value, sv.cvar_passes
    sv.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "sharded_inplace_timing_b200.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--shots", type=int, default=10000)
    ap.add_argument("--swaps", default="33:2,35:8,31:2v,32:2v,30:8v",
                    help="n:shards of the swap timings; a trailing v runs the shards round robin on the visible GPUs (HBM)")
    ap.add_argument("--run", default="36:8", help="n:shards of the full run ('' to skip)")
    args = ap.parse_args()
    out = {"card": card(), "visible_gpus": _native.device_count(), "swaps": [], "runs": []}
    print(json.dumps(out["card"]), flush=True)
    for spec in filter(None, args.swaps.split(",")):
        n, shards = spec.rstrip("v").split(":")
        rec = swap_case(int(n), int(shards), spec.endswith("v"), args.reps)
        print(json.dumps(rec), flush=True)
        out["swaps"].append(rec)
    for spec in filter(None, args.run.split(",")):
        n, shards = map(int, spec.split(":"))
        rec = evqe_run(n, shards, 2, args.shots)
        print(json.dumps(rec), flush=True)
        out["runs"].append(rec)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
