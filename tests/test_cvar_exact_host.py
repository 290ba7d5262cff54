"""Host logic of the exact (shot-free) CVaR route on CPU: argument checks, routing between ``Engine.expectation`` (alpha ~ 1 on
the operator evaluator) and ``Engine.cvar``, the coalescing key, the device split -- with a ``FakeEngine`` whose ``cvar`` is
the definition ``lower_tail_expectation_arrays(|psi|^2, E, alpha)`` -- and that definition against the reference's loop."""
import threading

import numpy as np
import pytest

from oracle import evqe_genome as og
from oracle import qiskit_semantics as oq
from queasars_b200 import expectation as ex
from queasars_b200 import primitives as pr
from queasars_b200.operators import SparsePauliOp
from tests.fake_engine import FakeEngine, _state
from tests.test_frontend_planner import build_circuit


class CvarFakeEngine(FakeEngine):
    def __init__(self, device=0, dtype="complex128"):
        super().__init__(device, dtype)
        self.calls = []

    def expectation(self, plans, params, ham):
        self.calls.append(("expectation", len(plans)))
        return super().expectation(plans, params, ham)

    def cvar(self, plans, params, ham, alpha):
        self.calls.append(("cvar", len(plans), alpha))
        n, xs, zs, cs = self._hams[ham.ham_id]
        if any(xs):
            raise ValueError("non-diagonal")
        table = oq.diagonal_table(n, [(z, c.real) for z, c in zip(zs, cs)])
        out = []
        for plan, vals in zip(plans, params):
            st = _state(self._plans[plan.plan_id], np.asarray(vals, dtype=np.float64).reshape(-1))
            out.append(ex.lower_tail_expectation_arrays(np.abs(st) ** 2, table, alpha))
        return np.asarray(out)


@pytest.fixture()
def fake_engines(monkeypatch):
    made = {}

    def get_engine(device=0, dtype="complex128"):
        return made.setdefault((device, dtype), CvarFakeEngine(device, dtype))

    monkeypatch.setattr(pr, "get_engine", get_engine)
    monkeypatch.setattr(pr._native, "device_count", lambda: 3)
    return made


def case(n, layers, seed):
    genome, values = og.random_individual(n, layers, True, seed)
    instr = og.individual_circuit(genome, values)
    return instr, list(values), build_circuit(instr, n)


def ising(n, seed=3):
    rng = np.random.default_rng(seed)
    terms = []
    for q in range(n):
        lab = ["I"] * n
        lab[n - 1 - q] = "Z"
        terms.append(("".join(lab), float(rng.normal())))
        lab[n - 1 - (q + 1) % n] = "Z"
        terms.append(("".join(lab), float(np.round(rng.normal()))))
    return terms


def oracle_value(instr, values, n, terms, alpha):
    probs = np.abs(oq.statevector(instr, n, values)) ** 2
    return ex.lower_tail_expectation_arrays(probs, oq.diagonal_table(n, oq.diag_terms_from_labels(terms)), alpha)


def calls(engines, kind):
    return [c for e in engines.values() for c in e.calls if c[0] == kind]


@pytest.mark.timeout(120)
@pytest.mark.parametrize("devices", [None, "all"])
def test_operator_evaluator_routes_by_alpha(fake_engines, devices):
    from queasars_b200.evaluators import B200OperatorSamplerCircuitEvaluator

    n = 5
    terms = ising(n)
    op = SparsePauliOp.from_list(terms)
    sampler = pr.B200SamplerV2(devices=devices)
    cases = [case(n, 2, s) for s in range(7)]
    circuits, params = [c for _, _, c in cases], [v for _, v, _ in cases]
    got = B200OperatorSamplerCircuitEvaluator(sampler, None, op, 0.5).evaluate_circuits(circuits, params)
    assert calls(fake_engines, "cvar") and not calls(fake_engines, "expectation")
    for g, (instr, values, _) in zip(got, cases):
        assert g == pytest.approx(oracle_value(instr, values, n, terms, 0.5), rel=1e-12)
    for e in fake_engines.values():
        e.calls.clear()
    got = B200OperatorSamplerCircuitEvaluator(sampler, None, op, 1.0).evaluate_circuits(circuits, params)
    assert calls(fake_engines, "expectation") and not calls(fake_engines, "cvar")
    table = oq.diagonal_table(n, oq.diag_terms_from_labels(terms))
    for g, (instr, values, _) in zip(got, cases):
        assert g == pytest.approx(float(np.dot(np.abs(oq.statevector(instr, n, values)) ** 2, table)), rel=1e-12)
    if devices == "all":  # the population is split over the device set
        assert sum(1 for e in fake_engines.values() if e.calls) > 1


def test_bitstring_evaluator_uses_cvar_at_every_alpha(fake_engines):
    from queasars_b200 import DiagonalEnergyBitstringEvaluator
    from queasars_b200.evaluators import B200BitstringCircuitEvaluator

    n = 4
    terms = ising(n, 8)
    diag = oq.diag_terms_from_labels(terms)
    bits = DiagonalEnergyBitstringEvaluator(n, [z for z, _ in diag], [c for _, c in diag])
    sampler = pr.B200SamplerV2()
    cases = [case(n, 2, 20 + s) for s in range(3)]
    for alpha in (0.3, 1.0):
        got = B200BitstringCircuitEvaluator(sampler, None, bits, alpha).evaluate_circuits([c for _, _, c in cases], [v for _, v, _ in cases])
        for g, (instr, values, _) in zip(got, cases):
            assert g == pytest.approx(oracle_value(instr, values, n, terms, alpha), rel=1e-12)
    assert [c[2] for c in calls(fake_engines, "cvar")] == [0.3, 1.0]
    assert not calls(fake_engines, "expectation")


def test_argument_checks(fake_engines):
    from queasars_b200 import BitstringEvaluator
    from queasars_b200.evaluators import B200BitstringCircuitEvaluator, B200OperatorSamplerCircuitEvaluator

    n = 4
    op = SparsePauliOp.from_list(ising(n))
    sampler = pr.B200SamplerV2()
    _, values, circ = case(n, 2, 1)
    with pytest.raises(ValueError):
        B200OperatorSamplerCircuitEvaluator(sampler, None, op, 0.0)
    with pytest.raises(ValueError):
        B200OperatorSamplerCircuitEvaluator(sampler, None, SparsePauliOp.from_list([("XIIZ", 1.0)]), 0.5)
    with pytest.raises(ValueError):
        B200BitstringCircuitEvaluator(sampler, None, BitstringEvaluator(n, lambda s: 0.0), 0.5)
    with pytest.raises(ValueError):
        sampler.cvar_values([circ], [values], op, 1.5)
    with pytest.raises(ValueError):
        sampler.cvar_values([circ], [values, values], op, 0.5)
    with pytest.raises(ValueError):
        sampler.cvar_values([circ], [values], SparsePauliOp.from_list([("XIIZ", 1.0)]), 0.5)
    with pytest.raises(ValueError):
        sampler.cvar_values([circ], [values], SparsePauliOp.from_list(ising(n + 1)), 0.5)
    assert sampler.cvar_values([], [], op, 0.5).shape == (0,)
    wide = pr.B200SamplerV2(shard_min_qubits=n)
    with pytest.raises(NotImplementedError):
        wide.cvar_values([circ], [values], op, 0.5)


def test_coalescing_key_keeps_alphas_apart(fake_engines):
    n = 4
    terms = ising(n)
    op = SparsePauliOp.from_list(terms)
    sampler = pr.B200SamplerV2()
    keys = []
    original = sampler._execute

    def spy(key, payloads):
        keys.append((key, len(payloads)))
        return original(key, payloads)

    sampler._execute = spy
    sampler._queue  # (built with the unwrapped method: route the queue through the spy as well)
    sampler._queue_obj._execute = spy
    cases = [case(n, 2, 40 + s) for s in range(8)]
    alphas = [0.2, 0.6] * 4
    results = [None] * len(cases)
    gate = threading.Barrier(len(cases))

    def work(i):
        gate.wait()
        instr, values, circ = cases[i]
        results[i] = sampler.cvar_values([circ], [values], op, alphas[i])[0]

    threads = [threading.Thread(target=work, args=(i,)) for i in range(len(cases))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for (instr, values, _), alpha, got in zip(cases, alphas, results):
        assert got == pytest.approx(oracle_value(instr, values, n, terms, alpha), rel=1e-12)
    for key, _ in keys:
        assert key[0] == "cvar" and key[3] in (0.2, 0.6) and key[4] == n
    assert {c[2] for c in calls(fake_engines, "cvar")} == {0.2, 0.6}
    assert sum(count for _, count in keys) == len(cases)


@pytest.mark.parametrize("seed", range(6))
def test_array_definition_matches_the_reference_loop(seed):
    rng = np.random.default_rng(seed)
    size = 1 << 9
    probs = rng.random(size) ** 4
    probs /= probs.sum()
    energies = rng.integers(-6, 6, size).astype(np.float64)  # heavily degenerate: the stop falls inside runs of ties
    if seed % 2:
        energies[rng.integers(0, size, 40)] = -0.0
        energies[energies == 0] = 0.0 if seed % 3 else -0.0
    for alpha in (0.01, 0.05, 0.25, 0.5, 0.9, 1.0):
        states = [(k, float(p), float(e)) for k, (p, e) in enumerate(zip(probs, energies))]
        want = oq.cvar_accumulate(states, alpha)
        got = ex.lower_tail_expectation_arrays(probs, energies, alpha)
        assert got == pytest.approx(want, rel=1e-12, abs=1e-12)
