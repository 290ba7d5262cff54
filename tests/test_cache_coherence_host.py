"""The primitives' memos on CPU against the oracle: the circuit cache keyed by ``id()``, the last-resolution memo of an identical
list, the Hamiltonian / observables cache and the evaluators' composed initial-state circuits -- on every route (Estimator,
Sampler, ``cvar_values``, ``top_states``, several observables, and the three evaluators with an initial-state circuit).  The
engine is the oracle-backed ``FakeEngine`` whose plans and Hamiltonians are forgotten when their handles die, as the native
ones are destroyed, so a memo that hands out a released handle fails here.

Out of scope, by design: the circuit fingerprint is ``(len(data), mutation counter)`` -- the parameter count for Qiskit
circuits -- a cheap guard, not a hash.  An edit that keeps ``len(data)`` and goes around the circuit's own methods, such as
``circ.data[i] = ...`` on a Qiskit circuit, is not noticed and the previous plan is used.
"""
import gc
import weakref

import numpy as np
import pytest

from oracle import evqe_genome as og
from oracle import qiskit_semantics as oq
from queasars_b200 import expectation as ex
from queasars_b200 import primitives as pr
from queasars_b200.circuit import QuantumCircuit
from queasars_b200.operators import SparsePauliOp
from tests.test_cvar_exact_host import CvarFakeEngine
from tests.test_frontend_planner import build_circuit
from tests.test_observables_host import ManyFakeEngine
from tests.test_top_states_host import TopFakeEngine, oracle_top

N = 5
SHOTS = 200
SEED = 13
ALPHA = 0.5


class RouteFakeEngine(CvarFakeEngine, ManyFakeEngine, TopFakeEngine):
    """Every route of the engine; a plan or Hamiltonian is dropped when its handle is released (Engine._release_*)."""

    def compile(self, gates, dtype=None, from_zero_state=True, cache=True, defer=True, drop_final_phases=False):
        handle = super().compile(gates, dtype, from_zero_state, cache, defer, drop_final_phases)
        weakref.finalize(handle, self._plans.pop, handle.plan_id, None)
        return handle

    def hamiltonian(self, operator, build_table=None):
        handle = super().hamiltonian(operator, build_table)
        weakref.finalize(handle, self._hams.pop, handle.ham_id, None)
        return handle


@pytest.fixture()
def engines(monkeypatch):
    made = {}
    monkeypatch.setattr(pr, "get_engine", lambda device=0, dtype="complex128": made.setdefault((device, dtype), RouteFakeEngine(device, dtype)))
    monkeypatch.setattr(pr._native, "device_count", lambda: 2)
    return made


class Case:
    """A circuit with its oracle instructions and parameter values by name (``QuantumCircuit.parameters`` order is by name)."""

    def __init__(self, seed, n=N, build=True):
        genome, values = og.random_individual(n, 2, True, seed)
        self.n, self.instr = n, og.individual_circuit(genome, values)
        rng = np.random.default_rng(seed)
        self.values = {name: float(v) for name, v in zip(oq.parameter_names(self.instr), rng.uniform(0, 6.28, len(values)))}
        if build:
            self.build()

    def build(self):
        self.circ = build_circuit(self.instr, self.n)

    def row(self):
        return [self.values[name] for name in oq.parameter_names(self.instr)]

    def state(self, prefix=()):
        instr = list(prefix) + self.instr
        return oq.statevector(instr, self.n, [self.values[name] for name in oq.parameter_names(instr)])


def bind_one(instr, name, value):
    """``instr`` with the parameter ``name`` bound to ``value`` (the oracle's form of a partial ``assign_parameters``)."""

    def bound(p):
        if p == name:
            return value
        return p[0] * value + p[2] if isinstance(p, tuple) and p[1] == name else p

    return [(g, q, tuple(bound(p) for p in ps)) for g, q, ps in instr]


def ising(n, seed):
    rng = np.random.default_rng(seed)
    terms = []
    for q in range(n):
        lab = ["I"] * n
        lab[n - 1 - q] = "Z"
        terms.append(("".join(lab), float(rng.normal())))
        lab[n - 1 - (q + 1) % n] = "Z"
        terms.append(("".join(lab), float(rng.normal())))
    return SparsePauliOp.from_list(terms)


def pauli_sum(n, seed):
    rng = np.random.default_rng(seed)
    return SparsePauliOp.from_list([("".join(rng.choice(list("IXYZ"), n)), float(rng.normal())) for _ in range(6)])


def table_of(op):
    return oq.diagonal_table(op.num_qubits, oq.diag_terms_from_labels(op.to_list()))


def every_route(est, smp, cases, op, observables):
    """Values of ``cases`` on every primitive route, next to the oracle's."""
    circuits, rows = [c.circ for c in cases], [c.row() for c in cases]
    states = [c.state() for c in cases]
    probs = [np.abs(s) ** 2 for s in states]
    table = table_of(op)
    uniforms = np.random.default_rng(SEED).random(SHOTS)  # the sampler's fresh default_rng(seed) per circuit
    pairs = {
        "estimator": (est.expectation_values(circuits, rows, op), [oq.estimator_expectation(s, op.to_list()) for s in states]),
        "estimator.run": ([float(r.data.evs) for r in est.run([(c, op, v) for c, v in zip(circuits, rows)]).result()],
                          [oq.estimator_expectation(s, op.to_list()) for s in states]),
        "observables": (est.expectation_values_many(circuits, rows, observables),
                        [[oq.estimator_expectation(s, o.to_list()) for o in observables] for s in states]),
        "sampler": (smp.sample_indices(circuits, rows, SHOTS), [oq.sample_indices(s, SHOTS, uniforms=uniforms) for s in states]),
        "cvar_values": (smp.cvar_values(circuits, rows, op, ALPHA), [ex.lower_tail_expectation_arrays(p, table, ALPHA) for p in probs]),
    }
    top = smp.top_states(circuits, rows, 4)
    for (idx, p), s in zip(top, states):
        want = oracle_top(s, 4)
        assert np.array_equal(idx, want[0]) and np.allclose(p, want[1], rtol=1e-12, atol=0), "top_states"
    for route, (got, want) in pairs.items():
        np.testing.assert_allclose(np.asarray(got, dtype=float), np.asarray(want, dtype=float), rtol=0, atol=1e-10, err_msg=route)


def primitives(devices, coalesce):
    return pr.B200EstimatorV2(devices=devices, coalesce=coalesce), pr.B200SamplerV2(devices=devices, coalesce=coalesce, seed=SEED)


@pytest.mark.timeout(300)
@pytest.mark.parametrize("old_alive", [False, True])
@pytest.mark.parametrize("devices,coalesce", [(None, False), ("all", True)])
def test_a_reused_id_gets_the_new_circuits_values(engines, monkeypatch, devices, coalesce, old_alive):
    """A circuit evaluated on every route goes away (or, stricter, stays alive) and a new circuit gets its ``id()``: the new
    circuit's values must be its own.  CPython hands a freed address to a later object, but not predictably, so the new circuit
    is given the old one's id through the ``id`` the primitives look up.  The new circuit is the old one's instructions in
    reverse order: same instruction and parameter counts, so the fingerprint alone cannot tell them apart."""
    import builtins

    alias = {}
    monkeypatch.setattr(pr, "id", lambda obj: alias.get(builtins.id(obj), builtins.id(obj)), raising=False)
    est, smp = primitives(devices, coalesce)
    op = ising(N, 1)
    observables = [op, pauli_sum(N, 2)]
    other = Case(999)
    for trial in range(3):
        old = Case(100 + trial)
        every_route(est, smp, [old, other, old], op, observables)
        every_route(est, smp, [old, other, old], op, observables)  # the identical list: the last-resolution memo
        new = Case(100 + trial, build=False)
        new.instr = new.instr[::-1]
        new.build()
        assert pr._circuit_fingerprint(new.circ) == pr._circuit_fingerprint(old.circ)
        old_id = builtins.id(old.circ)
        alias[builtins.id(new.circ)] = old_id
        if not old_alive:
            every_route(est, smp, [other], op, observables)  # (a coalescing worker lets go of the last list it ran)
            old_ref = weakref.ref(old.circ)
            del old
            gc.collect()
            assert old_ref() is None
        assert pr.id(new.circ) == old_id
        every_route(est, smp, [new, other, new], op, observables)
        every_route(est, smp, [new, other, new], op, observables)
        alias.clear()


@pytest.mark.timeout(300)
@pytest.mark.parametrize("edit", ["append", "assign_parameters", "coefficients"])
def test_guarded_edits_between_two_identical_calls(engines, edit):
    """Each edit the fingerprints promise to catch, between two calls with the same circuit list and operator objects."""
    est, smp = primitives("all", False)
    op = ising(N, 3)
    observables = [op, pauli_sum(N, 4)]
    a, b = Case(40), Case(41)
    cases = [a, b, a]
    every_route(est, smp, cases, op, observables)
    if edit == "append":
        a.circ.u(0.3, -0.7, 1.1, 2)
        a.circ.cx(2, 0)
        a.instr = a.instr + [("u", (2,), (0.3, -0.7, 1.1)), ("cx", (2, 0), ())]
    elif edit == "assign_parameters":
        first = a.circ.parameters[0]
        a.circ.assign_parameters({first: 0.25}, inplace=True)
        a.instr = bind_one(a.instr, first.name, 0.25)
        del a.values[first.name]
    else:
        op.coeffs[:] = op.coeffs * np.linspace(0.5, 2.0, op.coeffs.size)
    every_route(est, smp, cases, op, observables)


@pytest.mark.timeout(300)
@pytest.mark.parametrize("devices", [None, "all"])
def test_hamiltonian_cache_clear(engines, devices):
    """More than 64 operators per engine clear the Hamiltonian cache; the released device Hamiltonians are built again on their
    next use, and the circuits' memos, untouched, keep serving."""
    est, smp = primitives(devices, False)
    limit = 64 * len(est.engines)
    cases = [Case(60), Case(61)]
    ops = [ising(N, 200 + k) for k in range(limit + 6)]
    first_id = est.hamiltonian_for(ops[0]).ham_id
    for k, op in enumerate(ops):
        got = est.expectation_values([c.circ for c in cases], [c.row() for c in cases], op)
        want = [oq.estimator_expectation(c.state(), op.to_list()) for c in cases]
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-10, err_msg=f"operator {k}")
    assert len(est._ham_cache) < limit
    gc.collect()
    assert est.hamiltonian_for(ops[0]).ham_id != first_id  # released with the clear, built again
    for op in ops[:3] + ops[-2:]:
        every_route(est, smp, cases, op, [op, ops[1]])


def test_evaluators_with_an_initial_state_circuit(engines):
    """The three evaluators prepend an initial-state circuit (memoised per circuit object and fingerprint): values against the
    oracle of init + circuit, again after the circuit and after the initial-state circuit were edited in place."""
    from queasars_b200 import B200BitstringCircuitEvaluator, B200OperatorCircuitEvaluator, B200OperatorSamplerCircuitEvaluator
    from queasars_b200.bitstring_evaluation import DiagonalEnergyBitstringEvaluator

    op = ising(N, 5)
    table = table_of(op)
    init = QuantumCircuit(N)
    init_instr = []
    for q in range(N):
        init.h(q)
        init_instr.append(("h", (q,), ()))
    est, smp = pr.B200EstimatorV2(), pr.B200SamplerV2(seed=SEED)
    terms = op.to_list()
    z = [oq.pauli_label_to_masks(label)[1] for label, _ in terms]
    c = [float(np.real(coeff)) for _, coeff in terms]
    evaluators = {
        "operator": B200OperatorCircuitEvaluator(est, 0.0, op, initial_state_circuit=init),
        "operator_sampler_exact": B200OperatorSamplerCircuitEvaluator(smp, None, op, alpha=ALPHA, initial_state_circuit=init),
        "bitstring_shots": B200BitstringCircuitEvaluator(smp, SHOTS, DiagonalEnergyBitstringEvaluator(N, z, c), alpha=ALPHA, initial_state_circuit=init),
    }
    a, b = Case(70), Case(71)
    uniforms = np.random.default_rng(SEED).random(SHOTS)

    def want(name, case):
        state = case.state(init_instr)
        if name == "operator":
            return oq.estimator_expectation(state, terms)
        probs = np.abs(state) ** 2
        if name == "operator_sampler_exact":
            return ex.lower_tail_expectation_arrays(probs, table, ALPHA)
        states, counts = np.unique(oq.sample_indices(state, SHOTS, uniforms=uniforms), return_counts=True)
        return ex.lower_tail_expectation_arrays(counts / SHOTS, table[states], ALPHA)

    def check(what):
        for name, ev in evaluators.items():
            for _ in range(2):  # the second call re-uses the composed circuits and the last resolution
                got = ev.evaluate_circuits([a.circ, b.circ, a.circ], [a.row(), b.row(), a.row()])
                np.testing.assert_allclose(got, [want(name, x) for x in (a, b, a)], rtol=0, atol=1e-10, err_msg=f"{what}: {name}")

    check("as built")
    a.circ.ry(0.9, 1)
    a.instr = a.instr + [("ry", (1,), (0.9,))]
    check("circuit edited")
    init.rx(0.4, 3)
    init_instr.append(("rx", (3,), (0.4,)))
    check("initial-state circuit edited")
