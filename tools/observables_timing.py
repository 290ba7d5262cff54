"""Several observables per state (qb_evaluate_observables): one K-observable call against K single-observable calls on the same
circuits, and the share of the term-resolved reduction (expect_terms_tile_kernel, expect_terms_group_kernel,
reduce_term_partials_kernel, combine_observables_kernel) in the K-observable call.

Kernel times are GPU timestamps of torch.profiler (CUDA activities, CUPTI) summed per kernel name over the timed calls, in a
profiled pass of their own (sweep kernels that overlap on two streams are summed, not merged); end-to-end times are host clocks
around calls that end in a device synchronise (median of the repetitions), profiler off.  Both routes go through
B200EstimatorV2 without the coalescing queue; the single-observable route builds each observable's device form once, outside the
timed calls.

    python tools/observables_timing.py --out profiles/observables_timing_b200.json
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
from queasars_b200 import B200EstimatorV2  # noqa: E402
from queasars_b200 import expectation as ex  # noqa: E402
from queasars_b200.operators import SparsePauliOp  # noqa: E402
from tests.test_gpu_parity import tfim  # noqa: E402
from tools.cvar_timing import card, population, wall_ms  # noqa: E402

TERM_KERNELS = ("expect_terms_tile_kernel", "expect_terms_group_kernel", "reduce_term_partials_kernel", "combine_observables_kernel")
FAMILIES = ("sweep_kernel", "bind_kernel") + TERM_KERNELS


def label(n, paulis):
    lab = ["I"] * n
    for q, p in paulis.items():
        lab[n - 1 - q] = p
    return "".join(lab)


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
        for fam in FAMILIES:
            if fam in evt.key:
                out[fam] = out.get(fam, 0.0) + total / 1e3 / reps  # us -> ms per call
    return out


def case(name, ops, circuits, reps):
    est = B200EstimatorV2(device=0, coalesce=False)
    cs, vs = [c for c, _ in circuits], [v for _, v in circuits]
    many = lambda: est.expectation_values_many(cs, vs, ops)
    singles = lambda: [est.expectation_values(cs, vs, op) for op in ops]
    got = many()
    want = np.stack(singles(), axis=1)
    many_ms = wall_ms(many, reps)
    singles_ms = wall_ms(singles, max(1, reps // 3))
    ks = kernel_ms(many, reps)
    term_ms = sum(ks.get(k, 0.0) for k in TERM_KERNELS)
    n = ops[0].num_qubits
    handle = est.observables_for(ops)
    amp = 16 if est.dtype == "complex128" else 8
    return {
        "case": name, "n_qubits": n, "rows": len(cs), "observables": len(ops), "distinct_strings": handle.n_terms,
        "one_call_ms": many_ms, "single_observable_calls_ms": singles_ms, "speedup": singles_ms / many_ms,
        "max_rel_difference_to_single_route": float(np.max(np.abs(got - want) / np.maximum(1.0, np.abs(want)))),
        "kernel_ms_per_call": ks, "term_kernels_ms": term_ms, "term_kernels_share_of_call": term_ms / many_ms,
        # model: every tile sweep of groups reads each state once; one popcount / select / add per string and amplitude
        "tile_sweeps_state_bytes": len(cs) * (amp << max(n, 11)),
        "string_amplitude_ops": len(cs) * handle.n_terms * (1 << max(n, 11)),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=6)
    args = ap.parse_args()
    result = {"card": card(), "method": __doc__.split("\n\n")[1].replace("\n", " "), "cases": []}
    n = 20
    corr = [SparsePauliOp(label(n, {i: "Z"})) for i in range(n)]
    corr += [SparsePauliOp(label(n, {i: "Z", j: "Z"})) for i in range(n) for j in range(i + 1, n)]
    result["cases"].append(case("(a) 20q x 32, all <Z_i> and <Z_i Z_j>", corr, population(n, 32, 100), args.reps))
    n = 24
    parts = [SparsePauliOp.from_list(tfim(n))] + [SparsePauliOp(label(n, {i: "X"})) for i in range(n)]
    parts += [SparsePauliOp(label(n, {i: "Z"})) for i in range(n)]
    result["cases"].append(case("(b) 24q x 4, TFIM energy + <X_i> + <Z_i>", parts, population(n, 4, 300), args.reps))
    entry = json.load(open(os.path.join(ROOT, "tests", "golden", "jssp_hamiltonians.json")))["jssp_26q"]
    z, c = ex.merge_diagonal_terms(np.asarray(entry["z_masks"], dtype=np.uint64), np.asarray(entry["coeffs"], dtype=np.float64))
    energy = SparsePauliOp._raw(26, [0] * len(z), z.tolist(), c.tolist())
    # the energy and its terms split by weight (encoding penalties: one and two qubits; the rest: overlap / precedence)
    weight = np.array([bin(int(v)).count("1") for v in z])
    split = [SparsePauliOp._raw(26, [0] * int(m.sum()), z[m].tolist(), c[m].tolist()) for m in (weight <= 1, weight == 2, weight >= 3) if m.any()]
    result["cases"].append(case("(c) 26q x 2, JSSP energy + parts by term weight", [energy] + split, population(26, 2, 200), args.reps))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
