"""Sharded statevectors in complex64 against complex128 at the same width: both exchange kernels (swap_inplace_p2p_kernel, one
buffer per shard; swap_p2p_kernel, ping-pong into a second set) and one sweep of local gates per shard (``qb_apply_plan_device``
with an RY on every local qubit), alternated kernel by kernel and dtype by dtype in one process on the same raw shard buffers.

Times are host clocks around every shard's launch through the engine API, each ending in a device synchronise, joined over the
shards; median of `--reps` after one warm-up of each (kernel, dtype); the order alternates A B ... B A.  complex64 moves half the
bytes of complex128 (8 against 16 per amplitude): the record gives the time ratio complex64 / complex128 next to that byte ratio
of 0.5.  A case "n:shards" puts every shard on a GPU of its own (NVLink) and is recorded as not measured when the box has fewer
GPUs; "n:shardsv" runs the shards round robin on the visible GPUs, several virtual shards on one GPU exchanging through HBM.

    python tools/sharded_c64_timing.py --out profiles/sharded_c64_timing_b200.json
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
from queasars_b200 import QuantumCircuit  # noqa: E402
from queasars_b200 import _native  # noqa: E402
from queasars_b200 import gate_list as gl  # noqa: E402
from queasars_b200.primitives import get_engine  # noqa: E402

DTYPES = {"complex128": 16, "complex64": 8}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    rows = [[s.strip() for s in line.split(",")] for line in q.stdout.strip().splitlines()]
    return {"name": rows[0][0], "power_limit": rows[0][1], "gpus": len(rows), "power_limits": sorted({r[1] for r in rows})}


def free_bytes(devices):
    import torch

    return min(torch.cuda.mem_get_info(d)[0] for d in devices)


def case(n, shards, virtual, reps):
    from concurrent.futures import ThreadPoolExecutor

    n_dev = _native.device_count()
    g = int(math.log2(shards))
    nl = n - g
    rec = {"n": n, "shards": shards, "n_local": nl, "shard_GiB": {d: (a << nl) / 2**30 for d, a in DTYPES.items()}}
    if not virtual and n_dev < shards:
        rec["status"] = f"not measured: one GPU per shard (NVLink) needs {shards} GPUs, {n_dev} visible"
        return rec
    per_gpu = -(-shards // n_dev) if virtual else 1
    devices = sorted({r % n_dev for r in range(shards)})
    rec.update(gpus=len(devices), link="NVLink (one shard per GPU)" if per_gpu == 1 else f"HBM ({per_gpu} virtual shards per GPU)")
    need = 2 * sum(a << nl for a in DTYPES.values()) * per_gpu  # two sets per shard in both dtypes, resident together
    free = free_bytes(devices)
    if need + (2 << 30) > free:
        rec["status"] = f"not measured: {need / 2**30:.0f} GiB of shard buffers per GPU, {free / 2**30:.0f} GiB free"
        return rec
    engines = {d: [get_engine(r % n_dev, d) for r in range(shards)] for d in DTYPES}
    for d in DTYPES:
        for e in set(engines[d]):
            for dev in devices:
                e.enable_peer_access(dev)
    lp = list(range(nl - g, nl))
    circ = QuantumCircuit(nl)
    for q in range(nl):
        circ.ry(0.3 + 0.01 * q, q)
    state = {d: [] for d in DTYPES}
    spare = {d: [] for d in DTYPES}
    pool = ThreadPoolExecutor(max_workers=shards)
    try:
        plans = {}
        for d, amp in DTYPES.items():
            for e in engines[d]:
                state[d].append(e.device_alloc(amp << nl))
                spare[d].append(e.device_alloc(amp << nl))
            plans[d] = [e.compile(gl.from_circuit(circ), from_zero_state=False) for e in engines[d]]
            for r, e in enumerate(engines[d]):  # |0...0> on shard 0, zeros elsewhere: the RY sweeps keep every value finite
                e.apply_plan_device(plans[d][r], [], state[d][r], True, r << nl)
        rec["sweeps_per_plan"] = {d: plans[d][0].n_sweeps for d in DTYPES}

        def each(fn):  # every shard concurrently; returns when all of them completed
            list(pool.map(fn, range(shards)))

        def kernel(name, d):
            e = engines[d]
            if name == "inplace":
                return lambda r: (e[r].swap_global_inplace_p2p(d, nl, state[d], r, lp), e[r].synchronize())
            if name == "out_of_place":
                return lambda r: (e[r].swap_global_p2p(d, nl, state[d][r], spare[d], r, lp), e[r].synchronize())
            return lambda r: (e[r].apply_plan_device(plans[d][r], [], state[d][r], False, r << nl), e[r].synchronize())

        items = [(name, d) for name in ("inplace", "out_of_place", "sweep") for d in DTYPES]

        def timed(item):
            each(lambda r: engines[item[1]][r].synchronize())
            t0 = time.perf_counter()
            each(kernel(*item))
            return time.perf_counter() - t0

        for item in items:
            timed(item)  # warm-up
        times = {item: [] for item in items}
        for rep in range(reps):
            for item in (items if rep % 2 == 0 else items[::-1]):
                times[item].append(timed(item))
    finally:
        pool.shutdown(wait=True)
        for d in DTYPES:
            for r, e in enumerate(engines[d]):
                e.synchronize()
                for ptr in state[d][r:r + 1] + spare[d][r:r + 1]:
                    e.device_free(ptr)
    for name in ("inplace", "out_of_place", "sweep"):
        row = {}
        for d, amp in DTYPES.items():
            moved = ((1 - 2.0**-g) if name != "sweep" else 2 * rec["sweeps_per_plan"][d]) * (amp << nl) * per_gpu
            t = float(np.median(times[(name, d)]))
            row[d] = {"s": t, "all_s": times[(name, d)], "bytes_per_gpu": moved, "GBps_per_gpu": moved / t / 1e9}
        row["time_ratio_c64_over_c128"] = row["complex64"]["s"] / row["complex128"]["s"]
        row["byte_ratio_c64_over_c128"] = 0.5
        rec[name] = row
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "sharded_c64_timing_b200.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cases", default="32:2,34:8,31:2v,30:8v",
                    help="n:shards; a trailing v runs the shards round robin on the visible GPUs (HBM)")
    args = ap.parse_args()
    out = {"card": card(), "visible_gpus": _native.device_count(), "cases": []}
    print(json.dumps(out["card"]), flush=True)
    for spec in filter(None, args.cases.split(",")):
        n, shards = spec.rstrip("v").split(":")
        rec = case(int(n), int(shards), spec.endswith("v"), args.reps)
        print(json.dumps(rec), flush=True)
        out["cases"].append(rec)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
