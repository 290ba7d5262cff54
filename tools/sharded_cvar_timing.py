"""Exact CVaR of a sharded statevector (LocalShardedStatevector.cvar: the sort-free weighted select, cvar_select_kernel): circuit
run time against CVaR time, the number of select passes, bytes moved per pass against the measured 6.9 TB/s HBM read ceiling,
p and E cached in the spare shard buffer against recomputed on every pass, 10 000 shots for comparison, and the value against a
reference (the single-GPU Engine.cvar where the state fits one GPU, else the closed form of a product state).

Shards go round robin over the visible GPUs (several virtual shards per GPU when there are fewer GPUs than shards, as in the
tests); a case that does not fit the visible memory is reported as not measured.  Times are host clocks around calls that end in
a device synchronise (every native call of the select synchronises), median of `--reps`, after one warm-up call.

    python tools/sharded_cvar_timing.py --out profiles/sharded_cvar_timing_b200.json
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
from queasars_b200 import QuantumCircuit, _native  # noqa: E402
from queasars_b200 import gate_list as gl  # noqa: E402
from queasars_b200.operators import SparsePauliOp  # noqa: E402
from queasars_b200.primitives import get_engine  # noqa: E402
from tests.test_frontend_planner import build_circuit  # noqa: E402

READ_CEILING = 6.9e12  # B/s, measured HBM read ceiling of one B200 (profiles/r2_hbm_directional.json)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    name, power = [s.strip() for s in q.stdout.strip().split(",")]
    return {"name": name, "power_limit": power}


def ising_terms(n, seed, integer):
    """Z_i and Z_i Z_{i+1}, Z_i Z_{i+2} couplings; `integer`: small integer coefficients (a degenerate, JSSP-like spectrum)."""
    rng = np.random.default_rng(seed)
    z = [1 << q for q in range(n)] + [(1 << q) | (1 << ((q + d) % n)) for d in (1, 2) for q in range(n)]
    c = rng.integers(-2, 3, len(z)).astype(float) if integer else rng.normal(size=len(z))
    return z, [float(v) for v in c]


def median_time(fn, reps):
    fn()  # warm-up
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        times.append(time.perf_counter() - t0)
    return float(np.median(times)), out


def run_case(n, shards, kind, reps, shots):
    from queasars_b200.sharded import LocalShardedStatevector

    n_dev = _native.device_count()
    per_gpu = -(-shards // n_dev)
    need = 2 * (16 << (n - int(math.log2(shards)))) * per_gpu
    if n_dev < 1 or need > 0.85 * 180e9:
        return {"n": n, "shards": shards, "hamiltonian": kind, "status": f"not measured: {need / 2**30:.0f} GiB of shard buffers per GPU on {n_dev} GPU(s)"}
    engines = [get_engine(r % n_dev) for r in range(shards)]
    if kind == "product_sum_z":
        circ, values = QuantumCircuit(n), []
        for q in range(n):
            circ.ry(1.9, q)
        z, c = [1 << q for q in range(n)], [1.0] * n
    else:
        genome, values = og.random_individual(n, 6, True, 4242 + n)
        circ = build_circuit(og.individual_circuit(genome, values), n)
        z, c = ising_terms(n, 7, kind == "integer_ising_jssp_like")
    gates = gl.from_circuit(circ)
    rec = {"n": n, "shards": shards, "gpus": min(n_dev, shards), "hamiltonian": kind, "n_terms": len(z), "circuit_ops": len(gates.ops)}
    reference = {}
    if n <= 30 and kind != "product_sum_z":  # the single-GPU route still fits: its value and time
        eng = get_engine(0)
        ham = eng.hamiltonian(SparsePauliOp._raw(n, [0] * len(z), z, c), build_table=False)
        plan = eng.compile(gates, drop_final_phases=True)
        for alpha in (0.25, 1.0):
            t, v = median_time(lambda: eng.cvar([plan], [values], ham, alpha)[0], reps)
            reference[alpha] = (t, float(v))
        del ham, plan
    sv = LocalShardedStatevector(n, engines)

    def run():
        sv.reset()
        sv.run(gates, values)
        for e in set(engines):
            e.synchronize()

    rec["circuit_run_s"], _ = median_time(run, reps)
    amps_per_gpu = (1 << n) // shards * per_gpu
    rec["cases"] = []
    for alpha in (0.25, 1.0):
        for cache in (True, False):
            t, (value, stop) = median_time(lambda: sv.cvar(z, c, alpha, cache=cache), reps)
            passes = sv.cvar_passes
            # bytes per GPU: pass 1 reads the state (16 B / amplitude) and, cached, writes (p, E) (16 B); later passes read 16 B
            bytes_gpu = amps_per_gpu * 16 * (passes + (1 if cache else 0))
            row = {"alpha": alpha, "cache_p_E_in_spare": cache, "cvar_s": t, "passes": passes, "stop_index": stop, "value": value,
                   "bytes_per_gpu": bytes_gpu, "bytes_per_pass_per_gpu": amps_per_gpu * 16,
                   "share_of_read_ceiling": bytes_gpu / t / READ_CEILING, "cvar_over_circuit": t / rec["circuit_run_s"]}
            if alpha in reference:
                row["single_gpu_cvar_s"], row["single_gpu_value"] = reference[alpha]
                row["abs_diff_vs_single_gpu"] = abs(value - reference[alpha][1])
            if kind == "product_sum_z" and alpha < 1:
                s = math.sin(1.9 / 2) ** 2
                bound, acc, taken = alpha - (1e-8 + 1e-5 * alpha), 0.0, 0.0
                for j in range(n, -1, -1):
                    take = min(math.comb(n, j) * s**j * (1 - s) ** (n - j), bound - taken)
                    acc, taken = acc + take * (n - 2 * j), taken + take
                    if taken >= bound:
                        break
                row["closed_form_at_bound"] = acc / alpha
            rec["cases"].append(row)
    uniforms = np.random.default_rng(1).random(shots)
    rec["shots"] = shots
    rec["sample_s"], _ = median_time(lambda: sv.sample(shots, uniforms=uniforms), reps)
    sv.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "sharded_cvar_timing_b200.json"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--shots", type=int, default=10000)
    ap.add_argument("--cases", default="30:2:integer_ising_jssp_like,30:2:random_ising,35:8:product_sum_z,35:8:random_ising")
    args = ap.parse_args()
    out = {"card": card(), "visible_gpus": _native.device_count(), "read_ceiling_Bps": READ_CEILING, "results": []}
    for spec in args.cases.split(","):
        n, shards, kind = spec.split(":")
        rec = run_case(int(n), int(shards), kind, args.reps, args.shots)
        print(json.dumps(rec), flush=True)
        out["results"].append(rec)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
