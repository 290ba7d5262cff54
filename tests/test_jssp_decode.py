"""``jssp_decode.decode_start_times`` against the start times of the reference's own ``translate_result_bitstring`` for EVERY
basis state of small instances (the 4- and 8-qubit instances of the example notebooks and an 8-qubit variant) and a seeded
sample of the 26-qubit C4 instance.  Layouts and start times are stored in tests/golden/jssp_decode.json
(tests/golden/make_jssp_decode.py).  The stored layouts are checked against the energies of the reference encoder's own
Hamiltonian (tests/golden/jssp_hamiltonians.json).  When the reference package is installed, both are also compared with it
directly."""
import json
import os

import numpy as np
import pytest

from tests import reference_loop

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "jssp_decode.json")


@pytest.fixture(scope="module")
def decode_golden():
    with open(GOLDEN) as fh:
        return json.load(fh)


def _case(golden, spec, limit):
    spec = [[list(op) for op in job] for job in spec]
    (case,) = [c for c in golden.values() if c["spec"] == spec and c["limit"] == limit]
    return case


def _layout(case):
    from queasars_b200 import jssp_decode

    return [jssp_decode.OperationSlot(s["job"], s["operation"], s["start"], s["width"], tuple(s["values"])) for s in case["layout"]]


def _instance(ref, spec, limit):
    Machine, Operation, Job = ref["Machine"], ref["Operation"], ref["Job"]
    machines = {name: Machine(name=name) for name in sorted({m for job in spec for m, _ in job})}
    jobs = []
    for j, ops in enumerate(spec):
        jobs.append(Job(name=f"j{j}", operations=tuple(Operation(name=f"j{j}op{i}", machine=machines[m], processing_duration=d, job_name=f"j{j}") for i, (m, d) in enumerate(ops))))
    inst = ref["JobShopSchedulingProblemInstance"](name="inst", machines=tuple(machines.values()), jobs=tuple(jobs))
    return ref["JSSPDomainWallHamiltonianEncoder"](jssp_instance=inst, makespan_limit=limit, max_opt_value=100, opt_all_operations_share=0.19,
                                                   encoding_penalty=319, overlap_constraint_penalty=319, precedence_constraint_penalty=275)


def _reference_times(encoder, state, n):
    result = encoder.translate_result_bitstring(format(int(state), f"0{n}b"))
    row = []
    for job in encoder.jssp_instance.jobs:
        for op in result.schedule[job]:
            row.append(getattr(op, "start_time", None) if getattr(op, "is_scheduled", True) and hasattr(op, "start_time") else None)
    return [-1 if v is None else int(v) for v in row]


@pytest.mark.parametrize("spec,limit,exhaustive", [
    ([[("m0", 1), ("m1", 1)], [("m0", 1), ("m1", 1)]], 3, True),
    ([[("m0", 2), ("m1", 1)], [("m1", 1), ("m0", 2)]], 5, True),
    ([[("m0", 1), ("m1", 1), ("m2", 1), ("m3", 1), ("m4", 2)], [("m1", 2), ("m0", 1), ("m3", 2), ("m2", 1)], [("m2", 1), ("m4", 2), ("m0", 1), ("m1", 2)]], 8, False),
    ([[("m0", 2), ("m1", 1)], [("m0", 1), ("m1", 2)]], 5, True),
])
def test_vectorised_decode_matches_reference(decode_golden, spec, limit, exhaustive):
    from queasars_b200 import jssp_decode

    case = _case(decode_golden, spec, limit)
    layout = _layout(case)
    n = case["n_qubits"]
    assert sum(s.width for s in layout) == n
    states = np.asarray(case["states"], dtype=np.uint64)
    if exhaustive:
        np.testing.assert_array_equal(states, np.arange(1 << n, dtype=np.uint64))
    else:
        assert n == 26  # the C4 instance of SURVEY.md section 8d
    got = jssp_decode.decode_start_times(states, layout)
    np.testing.assert_array_equal(got, np.asarray(case["start_times"], dtype=np.int64))
    assert np.any(np.all(got >= 0, axis=1))
    if max(s.width for s in layout) > 1:  # one-qubit variables have no invalid pattern
        assert np.any(got < 0)
    if reference_loop.locate_reference() is not None:
        encoder = _instance(reference_loop.import_reference(), spec, limit)
        assert encoder.n_qubits == n
        assert [s._replace(values=tuple(int(v) for v in s.values)) for s in jssp_decode.layout_of(encoder)] == layout
        for row, state in zip(got, states):
            assert list(row) == _reference_times(encoder, state, n)


def _feasible(row, spec):
    """All operations scheduled, each after its predecessor in the job has finished, no two at once on one machine."""
    if np.any(row < 0):
        return False
    ops = [(j, m, d, int(t)) for (j, job), ts in zip(enumerate(spec), np.split(row, np.cumsum([len(job) for job in spec])[:-1])) for (m, d), t in zip(job, ts)]
    for a, b in zip(ops, ops[1:]):
        if a[0] == b[0] and b[3] < a[3] + a[2]:
            return False
    for i, a in enumerate(ops):
        for b in ops[i + 1:]:
            if a[1] == b[1] and a[3] < b[3] + b[2] and b[3] < a[3] + a[2]:
                return False
    return True


@pytest.mark.parametrize("name", ["4q", "8q"])
def test_decode_layout_matches_reference_hamiltonian(decode_golden, jssp_golden, name):
    """The reference encoder's Hamiltonian rates every feasible schedule below every other basis state (objective <= 100, each
    violated constraint costs >= 275).  So the states the stored layout decodes to feasible schedules must be exactly the ones
    below that gap, and the ground state must be among them."""
    from queasars_b200 import jssp_decode

    case = decode_golden[name]
    ham = jssp_golden[case["hamiltonian"]]
    assert ham["n_qubits"] == case["n_qubits"] and ham["makespan_limit"] == case["limit"]
    states = np.asarray(case["states"], dtype=np.uint64)
    z = np.asarray(ham["z_masks"], dtype=np.uint64)
    parity = np.bitwise_count(states[:, None] & z[None, :]) & 1
    energies = ((1 - 2 * parity.astype(np.float64)) * np.asarray(ham["coeffs"])).sum(axis=1)
    np.testing.assert_allclose(energies, ham["energies"], rtol=0, atol=1e-9)
    feasible = np.array([_feasible(row, case["spec"]) for row in jssp_decode.decode_start_times(states, _layout(case))])
    assert feasible.any() and not feasible.all()
    assert energies[feasible].max() < energies[~feasible].min()
    assert feasible[np.argmin(energies)]
