"""Exact (shot-free) CVaR(alpha) of diagonal Hamiltonians on the device (``qb_evaluate_cvar``, ``Engine.cvar``,
``B200SamplerV2.cvar_values`` and the sampler evaluators with ``sampler_shots=None``) against the definition
``expectation.lower_tail_expectation_arrays(|psi|^2, E, alpha)`` on the full distribution of the NumPy / C oracle state.

Knife edge: the device sums the running mass in a different order than ``np.cumsum``; where the oracle's running mass lies
within 1e-12 of the stop bound ``alpha - isclose tolerance``, the value of the neighbouring stop index is accepted too (the
sampler tests' "<= 1 boundary flip" rule).  ``EDGES`` counts those cases; the module reports it at the end.
"""
import numpy as np
import pytest

from oracle import c_oracle
from oracle import evqe_genome as og
from oracle import qiskit_semantics as oq
from queasars_b200 import expectation as ex
from queasars_b200 import gate_list as gl
from queasars_b200.operators import SparsePauliOp
from tests.test_frontend_planner import build_circuit
from tests.test_gpu_parity import random_ising

pytestmark = pytest.mark.gpu

ALPHAS = (0.05, 0.25, 0.5, 0.9, 1.0)
EDGES = {"checked": 0, "knife_edge": 0}


def evqe_case(n, layers, seed):
    genome, values = og.random_individual(n, layers, True, seed)
    instr = og.individual_circuit(genome, values)
    return instr, list(values), build_circuit(instr, n)


def probs_of(instr, n, values):
    if n < 16:
        return np.abs(oq.statevector(instr, n, values)) ** 2
    _, state = c_oracle.evaluate(instr, n, values, None, np.empty(1 << n, dtype=np.complex128))
    return state.real**2 + state.imag**2


def accepted_values(probs, energies, alpha):
    """The reference value and, at a knife edge, the values of the neighbouring stop indices."""
    want = ex.lower_tail_expectation_arrays(probs, energies, alpha)
    ps, es = probs, energies
    if not ex._close(alpha, 1):
        order = np.argsort(energies, kind="stable")
        ps, es = probs[order], energies[order]
    cum = np.cumsum(ps)
    bound = alpha - (1e-8 + 1e-5 * alpha)
    before = np.concatenate(([0.0], cum[:-1]))
    # every stop index some summation order within 1e-12 of cumsum could pick
    stops = np.nonzero((before < bound + 1e-12) & (cum >= bound - 1e-12))[0]
    EDGES["checked"] += 1
    if stops.size <= 1:
        return [want]
    EDGES["knife_edge"] += 1
    pe = np.concatenate(([0.0], np.cumsum(ps * es)))
    return [want] + [(pe[k] + min(alpha - before[k], ps[k]) * es[k]) / alpha for k in stops]


def assert_cvar(got, probs, energies, alpha, rtol):
    cands = accepted_values(probs, energies, alpha)
    scale = max(1.0, abs(cands[0]))
    err = min(abs(got - c) for c in cands) / scale
    assert err <= rtol, f"alpha={alpha}: got {got!r}, oracle {cands[0]!r} (rel {err:.2e})"


@pytest.fixture(scope="module", autouse=True)
def report_edges():
    yield
    print(f"\nexact CVaR: {EDGES['knife_edge']} knife-edge stops in {EDGES['checked']} oracle comparisons")


@pytest.fixture(scope="module")
def engine():
    from queasars_b200.engine import Engine

    return Engine(device=0, dtype="complex128")


def diag_op(n, z, c):
    return SparsePauliOp._raw(n, [0] * len(z), [int(v) for v in z], [float(v) for v in c])


def jssp_op(entry):
    z, c = ex.merge_diagonal_terms(np.asarray(entry["z_masks"], dtype=np.uint64), np.asarray(entry["coeffs"], dtype=np.float64))
    return diag_op(int(entry["n_qubits"]), z, c), list(zip(z.tolist(), c.tolist()))


# ------------------------------------------------------------------------------------ random EVQE individuals
@pytest.mark.parametrize("n", [4, 12, 20])
def test_random_individuals_against_the_oracle(engine, n):
    terms = random_ising(n)
    diag_terms = oq.diag_terms_from_labels(terms)
    table = oq.diagonal_table(n, diag_terms) if n < 20 else c_oracle.diag_table(n, diag_terms)
    ham = engine.hamiltonian(SparsePauliOp.from_list(terms), build_table=False)
    cases = [evqe_case(n, 2 + s % 5, 7000 + 31 * n + s) for s in range(32)]
    plans = [engine.compile(gl.from_circuit(c), drop_final_phases=True) for _, _, c in cases]
    params = [v for _, v, _ in cases]
    probs = [probs_of(instr, n, values) for instr, values, _ in cases]
    for alpha in ALPHAS:
        got = engine.cvar(plans, params, ham, alpha)
        for g, p in zip(got, probs):
            assert_cvar(g, p, table, alpha, 1e-10)


# ------------------------------------------------------------------------------------ JSSP golden Hamiltonians (degenerate)
@pytest.mark.parametrize("name", ["jssp_4q", "jssp_5q", "jssp_8q", "jssp_12q", "jssp_unit_test"])
def test_jssp_hamiltonians_entangled_states(engine, jssp_golden, name):
    op, diag_terms = jssp_op(jssp_golden[name])
    n = op.num_qubits
    table = oq.diagonal_table(n, diag_terms)
    ham = engine.hamiltonian(op, build_table=False)
    cases = [evqe_case(n, 3 + s % 3, 900 + s) for s in range(8)]
    plans = [engine.compile(gl.from_circuit(c), drop_final_phases=True) for _, _, c in cases]
    probs = [probs_of(instr, n, values) for instr, values, _ in cases]
    for alpha in ALPHAS:
        got = engine.cvar(plans, [v for _, v, _ in cases], ham, alpha)
        for g, p in zip(got, probs):
            assert_cvar(g, p, table, alpha, 1e-10)


def test_jssp_26q_entangled_state(engine, jssp_golden):
    op, diag_terms = jssp_op(jssp_golden["jssp_26q"])
    n = 26
    table = c_oracle.diag_table(n, diag_terms)
    ham = engine.hamiltonian(op, build_table=False)
    instr, values, circ = evqe_case(n, 4, 26)
    state = np.empty(1 << n, dtype=np.complex128)
    c_oracle.evaluate(instr, n, values, None, state)
    probs = state.real**2 + state.imag**2
    del state
    plan = engine.compile(gl.from_circuit(circ), drop_final_phases=True)
    for alpha in (0.05, 0.5, 1.0):
        assert_cvar(engine.cvar([plan], [values], ham, alpha)[0], probs, table, alpha, 1e-10)


# ------------------------------------------------------------------------------------ special states and dtypes
@pytest.mark.parametrize("name", ["jssp_5q", "jssp_12q"])
def test_basis_states_give_their_energy(engine, jssp_golden, name):
    from queasars_b200 import QuantumCircuit

    op, diag_terms = jssp_op(jssp_golden[name])
    n = op.num_qubits
    ham = engine.hamiltonian(op, build_table=False)
    rng = np.random.default_rng(n)
    states = [0, (1 << n) - 1] + [int(k) for k in rng.integers(0, 1 << n, 6)]
    plans = []
    for k in states:
        circ = QuantumCircuit(n)
        for q in range(n):
            if (k >> q) & 1:
                circ.x(q)
            else:
                circ.id(q)
        plans.append(engine.compile(gl.from_circuit(circ), drop_final_phases=True))
    for alpha in ALPHAS:
        got = engine.cvar(plans, [[] for _ in plans], ham, alpha)
        for g, k in zip(got, states):
            assert g == pytest.approx(oq.diagonal_energy(k, diag_terms), rel=1e-12, abs=1e-12)


@pytest.mark.parametrize("n", [12, 20])
def test_complex64_against_the_complex128_oracle(n):
    from queasars_b200.engine import Engine

    eng = Engine(device=0, dtype="complex64")
    terms = random_ising(n, 5)
    table = c_oracle.diag_table(n, oq.diag_terms_from_labels(terms))
    ham = eng.hamiltonian(SparsePauliOp.from_list(terms), build_table=False)
    cases = [evqe_case(n, 3, 4000 + s) for s in range(8)]
    plans = [eng.compile(gl.from_circuit(c), drop_final_phases=True) for _, _, c in cases]
    probs = [probs_of(instr, n, values) for instr, values, _ in cases]
    for alpha in ALPHAS:
        got = eng.cvar(plans, [v for _, v, _ in cases], ham, alpha)
        for g, p in zip(got, probs):
            want = ex.lower_tail_expectation_arrays(p, table, alpha)
            assert abs(g - want) <= 1e-4 * max(1.0, abs(want))


# ------------------------------------------------------------------------------------ determinism
def test_bit_identical_across_calls_and_batch_compositions(engine):
    n = 16
    ham = engine.hamiltonian(SparsePauliOp.from_list(random_ising(n, 9)), build_table=False)
    cases = [evqe_case(n, 2 + s % 4, 300 + s) for s in range(32)]
    plans = [engine.compile(gl.from_circuit(c), drop_final_phases=True) for _, _, c in cases]
    params = [v for _, v, _ in cases]
    for alpha in (0.25, 1.0):
        a = engine.cvar(plans, params, ham, alpha)
        b = engine.cvar(plans, params, ham, alpha)
        assert a.tobytes() == b.tobytes()
        for i in (0, 13, 31):
            alone = engine.cvar([plans[i]], [params[i]], ham, alpha)[0]
            assert alone.tobytes() == a[i].tobytes()


def test_batch_larger_than_the_workspace_is_chunked():
    from queasars_b200.engine import Engine

    n = 16  # 1 MiB states, 1.25 MiB of order data: a 24 MiB workspace holds 22 states next to it
    eng = Engine(device=0, workspace_limit=24 << 20)
    ham = eng.hamiltonian(SparsePauliOp.from_list(random_ising(n, 11)), build_table=False)
    cases = [evqe_case(n, 3, 600 + s) for s in range(48)]
    plans = [eng.compile(gl.from_circuit(c), drop_final_phases=True) for _, _, c in cases]
    params = [v for _, v, _ in cases]
    whole = eng.cvar(plans, params, ham, 0.5)
    parts = np.concatenate([eng.cvar(plans[lo : lo + 8], params[lo : lo + 8], ham, 0.5) for lo in range(0, 48, 8)])
    assert whole.tobytes() == parts.tobytes()


def test_order_data_larger_than_the_workspace_is_refused():
    from queasars_b200 import _native
    from queasars_b200.engine import Engine

    n = 16  # one 1 MiB state fits, the 1.25 MiB of order data next to it does not
    eng = Engine(device=0, workspace_limit=(1 << 20) + (64 << 10))
    ham = eng.hamiltonian(SparsePauliOp.from_list(random_ising(n, 11)), build_table=False)
    _, values, circ = evqe_case(n, 2, 1)
    with pytest.raises(_native.QbError, match="bytes") as err:
        eng.cvar([eng.compile(gl.from_circuit(circ))], [values], ham, 0.5)
    assert err.value.code == _native.QB_ERR_MEMORY


def test_alpha_one_needs_no_sorted_order():
    from queasars_b200.engine import Engine

    n = 16  # 0.5 MiB of energies and a 1 MiB state fit 1.75 MiB; the 1.25 MiB of sorted order data with them would not
    eng = Engine(device=0, workspace_limit=(1 << 20) + (768 << 10))
    terms = random_ising(n, 11)
    ham = eng.hamiltonian(SparsePauliOp.from_list(terms), build_table=False)
    instr, values, circ = evqe_case(n, 2, 1)
    got = eng.cvar([eng.compile(gl.from_circuit(circ), drop_final_phases=True)], [values], ham, 1.0)[0]
    assert_cvar(got, probs_of(instr, n, values), c_oracle.diag_table(n, oq.diag_terms_from_labels(terms)), 1.0, 1e-10)


@pytest.mark.parametrize("narrower", [False, True])
def test_mixed_widths_in_a_split_list_are_refused(narrower):
    from queasars_b200 import _native
    from queasars_b200.engine import Engine

    # 1 MiB states next to 1.25 MiB of order data in a 24 MiB workspace: the list is split after 22 states, so the 4 plans of
    # another width form a chunk of their own, launched against order data built for the first plan's width
    n = 16
    eng = Engine(device=0, workspace_limit=24 << 20)
    ham = eng.hamiltonian(SparsePauliOp.from_list(random_ising(n, 11)), build_table=False)
    other = n - 1 if narrower else n + 1
    cases = [evqe_case(n, 2, 700 + s) for s in range(22)] + [evqe_case(other, 2, 800 + s) for s in range(4)]
    plans = [eng.compile(gl.from_circuit(c), drop_final_phases=True) for _, _, c in cases]
    eng.cvar(plans[:1], [cases[0][1]], ham, 0.5)  # the order data exists
    for alpha in (0.5, 1.0):
        with pytest.raises(_native.QbError) as err:
            eng.cvar(plans, [v for _, v, _ in cases], ham, alpha)
        assert err.value.code == _native.QB_ERR_INVALID


def test_length_mismatch_is_a_value_error(engine):
    from queasars_b200 import QuantumCircuit

    n = 6
    ham = engine.hamiltonian(SparsePauliOp.from_list(random_ising(n, 2)), build_table=False)
    fixed = QuantumCircuit(n)
    fixed.x(0)
    plain = engine.compile(gl.from_circuit(fixed))
    _, values, circ = evqe_case(n, 2, 3)
    param = engine.compile(gl.from_circuit(circ))
    with pytest.raises(ValueError):
        engine.cvar([plain, plain], [[]], ham, 0.5)
    with pytest.raises(ValueError):
        engine.cvar([param, param], [values], ham, 0.5)


# ------------------------------------------------------------------------------------ evaluators
@pytest.mark.parametrize("name", ["jssp_12q"])
def test_evaluators_with_exact_mode(jssp_golden, name):
    from queasars_b200 import (B200BitstringCircuitEvaluator, B200OperatorSamplerCircuitEvaluator, B200SamplerV2,
                               DiagonalEnergyBitstringEvaluator, QuantumCircuit)

    op, diag_terms = jssp_op(jssp_golden[name])
    n = op.num_qubits
    table = oq.diagonal_table(n, diag_terms)
    z, c = zip(*diag_terms)
    sampler = B200SamplerV2(device=0, seed=3)
    cases = [evqe_case(n, 3, 50 + s) for s in range(6)]
    circuits, params = [cc for _, _, cc in cases], [v for _, v, _ in cases]
    probs = [probs_of(instr, n, values) for instr, values, _ in cases]
    init = QuantumCircuit(n)
    for q in range(0, n, 3):
        init.x(q)
    init_instr = [("u", (q,), (np.pi, 0.0, np.pi)) for q in range(0, n, 3)]
    probs_init = [np.abs(oq.statevector(init_instr + list(instr), n, values)) ** 2 for instr, values, _ in cases]
    for alpha in ALPHAS:
        got = B200OperatorSamplerCircuitEvaluator(sampler, None, op, alpha).evaluate_circuits(circuits + [None], params + [[0.0]])
        assert len(got) == len(cases)
        for g, p in zip(got, probs):
            if ex._close(alpha, 1):  # sum p E, as the sampled branch
                assert g == pytest.approx(float(np.dot(p, table)), rel=1e-10, abs=1e-10)
            else:
                assert_cvar(g, p, table, alpha, 1e-10)
        bit = B200BitstringCircuitEvaluator(sampler, None, DiagonalEnergyBitstringEvaluator(n, z, c), alpha)
        for g, p in zip(bit.evaluate_circuits(circuits, params), probs):
            assert_cvar(g, p, table, alpha, 1e-10)
        with_init = B200OperatorSamplerCircuitEvaluator(sampler, None, op, alpha, initial_state_circuit=init)
        for g, p in zip(with_init.evaluate_circuits(circuits, params), probs_init):
            if ex._close(alpha, 1):
                assert g == pytest.approx(float(np.dot(p, table)), rel=1e-10, abs=1e-10)
            else:
                assert_cvar(g, p, table, alpha, 1e-10)
    assert B200OperatorSamplerCircuitEvaluator(sampler, None, op, 0.5).evaluate_circuits([], []) == []


def test_device_set_gives_the_single_device_values(jssp_golden):
    from queasars_b200 import B200BitstringCircuitEvaluator, B200OperatorSamplerCircuitEvaluator, B200SamplerV2, DiagonalEnergyBitstringEvaluator

    op, diag_terms = jssp_op(jssp_golden["jssp_12q"])
    n = op.num_qubits
    z, c = zip(*diag_terms)
    cases = [evqe_case(n, 2 + s % 4, 80 + s) for s in range(24)]
    circuits, params = [cc for _, _, cc in cases], [v for _, v, _ in cases]
    single, multi = B200SamplerV2(device=0), B200SamplerV2(devices="all")
    for alpha in (0.5, 1.0):
        a = B200OperatorSamplerCircuitEvaluator(single, None, op, alpha).evaluate_circuits(circuits, params)
        b = B200OperatorSamplerCircuitEvaluator(multi, None, op, alpha).evaluate_circuits(circuits, params)
        assert np.asarray(a).tobytes() == np.asarray(b).tobytes()
        bs = DiagonalEnergyBitstringEvaluator(n, z, c)
        a = B200BitstringCircuitEvaluator(single, None, bs, alpha).evaluate_circuits(circuits, params)
        b = B200BitstringCircuitEvaluator(multi, None, bs, alpha).evaluate_circuits(circuits, params)
        assert np.asarray(a).tobytes() == np.asarray(b).tobytes()


# ------------------------------------------------------------------------------------ errors
def test_errors(engine):
    from queasars_b200 import B200BitstringCircuitEvaluator, B200OperatorSamplerCircuitEvaluator, B200SamplerV2, BitstringEvaluator, _native

    n = 6
    sampler = B200SamplerV2(device=0)
    with pytest.raises(ValueError):
        B200OperatorSamplerCircuitEvaluator(sampler, None, SparsePauliOp.from_list([("XIIIIZ", 1.0), ("ZZIIII", 0.5)]), 0.5)
    with pytest.raises(ValueError):
        B200BitstringCircuitEvaluator(sampler, None, BitstringEvaluator(n, lambda s: float(s.count("1"))), 0.5)
    with pytest.raises(ValueError):
        B200OperatorSamplerCircuitEvaluator(sampler, None, SparsePauliOp.from_list([("ZZIIII", 0.5)]), 0.0)
    mixed = engine.hamiltonian(SparsePauliOp.from_list([("XIIIIZ", 1.0), ("ZZIIII", 0.5)]))
    _, values, circ = evqe_case(n, 2, 5)
    with pytest.raises(_native.QbError):
        engine.cvar([engine.compile(gl.from_circuit(circ))], [values], mixed, 0.5)
