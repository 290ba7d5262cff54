"""Generate tests/golden/jssp_decode.json: domain-wall layouts and decoded start times for tests/test_jssp_decode.py.

    python tests/golden/make_jssp_decode.py

For every instance the file holds the job spec, the makespan limit, the layout of the start-time variables and, for a
set of basis states, the start time of every operation (-1 = unscheduled).

Layout: ``JSSPDomainWallHamiltonianEncoder`` gives each operation, jobs in instance order and operations in job order, one
domain-wall variable on consecutive qubits. Its values are the start times from the sum of the durations before the
operation in its job up to the makespan limit minus the durations from the operation on, and it takes one qubit fewer than
it has values. The test checks these layouts against the energies of the original encoder's own Hamiltonian
(jssp_hamiltonians.json, written by make_golden.py from the reference package). When the reference package is installed it
also compares them with the encoder's ``_operation_start_variables``.

Rows: ``jssp_decode.decode_start_times`` on these layouts. The decoder was checked state by state against the reference's
``translate_result_bitstring`` on these instances. The test repeats that comparison when the reference package is installed.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..", "..")))

from queasars_b200 import jssp_decode  # noqa: E402

CASES = {
    # examples/evqe_jssp_small_examples.ipynb cells 4+8 (jssp_4q of jssp_hamiltonians.json)
    "4q": {"spec": [[["m0", 1], ["m1", 1]], [["m0", 1], ["m1", 1]]], "limit": 3, "hamiltonian": "jssp_4q"},
    # 8 qubits, the second job in the opposite machine order
    "8q_crossed": {"spec": [[["m0", 2], ["m1", 1]], [["m1", 1], ["m0", 2]]], "limit": 5, "hamiltonian": None},
    # examples/using_the_ibm_runtime.ipynb cells 2+6 (jssp_8q)
    "8q": {"spec": [[["m0", 2], ["m1", 1]], [["m0", 1], ["m1", 2]]], "limit": 5, "hamiltonian": "jssp_8q"},
    # SURVEY.md section 8d, config C4 (jssp_26q): a seeded sample of basis states plus domain-valid codes
    "26q": {"spec": [[["m0", 1], ["m1", 1], ["m2", 1], ["m3", 1], ["m4", 2]], [["m1", 2], ["m0", 1], ["m3", 2], ["m2", 1]],
                     [["m2", 1], ["m4", 2], ["m0", 1], ["m1", 2]]], "limit": 8, "hamiltonian": "jssp_26q"},
}


def layout(spec, limit):
    slots, qubit = [], 0
    for j, ops in enumerate(spec):
        durations = [d for _, d in ops]
        for i in range(len(ops)):
            values = list(range(sum(durations[:i]), limit - sum(durations[i:]) + 1))
            slots.append({"job": f"j{j}", "operation": f"j{j}op{i}", "start": qubit, "width": len(values) - 1, "values": values})
            qubit += len(values) - 1
    return slots


def states_for(slots):
    n = sum(s["width"] for s in slots)
    if n <= 12:
        return np.arange(1 << n, dtype=np.uint64)
    states = np.random.default_rng(0).integers(0, 1 << n, size=300, dtype=np.uint64)
    # all walls at zero, then the walls of the first k variables half way up: valid codes among the sample
    valid = [0]
    for s in slots:
        valid.append(valid[-1] | (((1 << (s["width"] // 2)) - 1) << s["start"]))
    return np.concatenate([states, np.asarray(valid, dtype=np.uint64)])


def main():
    out = {}
    for name, case in CASES.items():
        slots = layout(case["spec"], case["limit"])
        states = states_for(slots)
        rows = jssp_decode.decode_start_times(states, [jssp_decode.OperationSlot(s["job"], s["operation"], s["start"], s["width"], tuple(s["values"])) for s in slots])
        out[name] = dict(case, n_qubits=sum(s["width"] for s in slots), layout=slots, states=[int(k) for k in states], start_times=rows.tolist())
    with open(os.path.join(HERE, "jssp_decode.json"), "w") as fh:
        json.dump(out, fh, separators=(",", ":"))
    print("wrote jssp_decode.json")


if __name__ == "__main__":
    main()
