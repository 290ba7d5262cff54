"""B200 circuit evaluators: drop-ins for the three evaluator classes of
/root/reference/queasars/circuit_evaluation/circuit_evaluation.py behind the same interface

    evaluate_circuits(circuits: list[QuantumCircuit], parameter_values: list[list[float]]) -> list[float]
    n_qubits -> int                                                        (circuit_evaluation.py:62-87)

with the same constructor argument order, the same ``ValueError`` conditions (alpha outside (0, 1],
non-SparsePauliOp operator on the sampler route, qubit-count mismatch of ``initial_state_circuit``) and the same
result semantics, but evaluating the whole list in one batched GPU submission instead of one primitive pub
per circuit.  Inputs are never mutated; outputs are fresh Python floats.

``sampler_shots=None`` on the two sampler evaluators means exact values: CVaR(alpha) of the full distribution |psi|^2 of the
statevector instead of a shot histogram (``B200SamplerV2.cvar_values``; with alpha close to 1 the operator evaluator returns
sum_k |psi_k|^2 E(k)), so the objective carries no shot noise.  It needs a diagonal energy on the device: a ``SparsePauliOp`` of
Z terms, or a bitstring evaluator exposing ``diagonal_terms``.

Differences that are deliberate and documented in DESIGN.md:
  * the first constructor argument must be a ``B200EstimatorV2`` / ``B200SamplerV2`` (it carries device,
    dtype and seed); any other primitive type raises ``TypeError`` -- to drive a foreign primitive use the
    reference's own evaluators, to drive the B200 engine through the reference's own evaluators hand them the
    B200 primitives;
  * sampled bitstrings are always formatted with ``n_qubits`` characters (the reference inherits upstream
    ``QuasiDistribution.binary_probabilities()``'s pad-to-longest-observed quirk, which can make
    ``BitstringEvaluator`` raise on short strings: expectation_calculation.py:96, bitstring_evaluation.py:29-32).
"""
from __future__ import annotations

from abc import ABC, abstractmethod
from typing import Optional

import numpy as np

from . import expectation as ex
from .containers import QuasiDistribution
from .engine import operator_terms
from .primitives import B200EstimatorV2, B200SamplerV2, _circuit_fingerprint


class CircuitEvaluatorException(Exception):
    """Raised when a circuit evaluation fails (circuit_evaluation.py:90-91)."""


try:  # subclass the reference ABC when it is importable so isinstance() checks in user code keep working
    from queasars.circuit_evaluation.circuit_evaluation import BaseCircuitEvaluator as _ReferenceBase  # type: ignore
except Exception:  # pragma: no cover - reference package absent
    _ReferenceBase = None


class BaseCircuitEvaluator(ABC):
    @abstractmethod
    def evaluate_circuits(self, circuits: list, parameter_values: list[list[float]]) -> list[float]:
        ...

    @property
    @abstractmethod
    def n_qubits(self) -> int:
        ...


if _ReferenceBase is not None:
    _ReferenceBase.register(BaseCircuitEvaluator)


def measure_quasi_distributions(circuits: list, parameter_values: list[list[float]], sampler, shots: Optional[int], *,
                                max_states: int = 1024) -> list[QuasiDistribution]:
    """Same contract as circuit_evaluation.py:29-59.  With a ``B200SamplerV2`` the ``measure_all`` copy and the
    per-pub primitive round trip are skipped (sampling the full register *is* measure_all); any other
    SamplerV2 goes through the generic pub path exactly like the reference.

    ``shots=None`` with a ``B200SamplerV2``: no sampling -- every distribution holds the exact probabilities of the
    ``max_states`` most probable basis states of its circuit's state (``B200SamplerV2.top_states``; ties in ascending basis
    index), with ``shots=None``.  The default of 1024 is the most entries a 1024-shot distribution can hold."""
    if isinstance(sampler, B200SamplerV2):
        pairs = [(c, p) for c, p in zip(circuits, parameter_values) if c is not None and p is not None]
        if shots is None:
            tops = sampler.top_states([c for c, _ in pairs], [p for _, p in pairs], max_states)
            return [QuasiDistribution({int(k): float(v) for k, v in zip(idx, probs)}, shots=None) for idx, probs in tops]
        idx = sampler.sample_indices([c for c, _ in pairs], [p for _, p in pairs], shots)
        out = []
        for row in idx:
            vals, cnts = np.unique(row, return_counts=True)
            out.append(QuasiDistribution({int(v): int(c) / shots for v, c in zip(vals, cnts)}, shots=shots))
        return out
    measured = [circuit.measure_all(inplace=False) for circuit in circuits]
    pubs = tuple((c, p) for c, p in zip(measured, parameter_values) if c is not None and p is not None)
    result = sampler.run(pubs=pubs, shots=shots).result()
    return [
        QuasiDistribution({state: count / shots for state, count in res.data["meas"].get_counts().items()}, shots=shots)
        for res in result
    ]


def _check_initial_state(initial_state_circuit, n_qubits: int, what: str) -> None:
    if initial_state_circuit is not None and initial_state_circuit.num_qubits != n_qubits:
        raise ValueError(
            f"The amount of qubits in the initial state circuit ({initial_state_circuit.num_qubits} "
            + f"does not match {what} ({n_qubits})"
        )


class _WithInitialState:
    _initial_state_circuit = None

    def _prepend(self, circuits: list) -> list:
        """``initial_state_circuit.compose(circuit, inplace=False)`` per circuit (circuit_evaluation.py:148-149),
        memoised per circuit object so the plan cache (keyed by identity) still hits on repeated calls."""
        if self._initial_state_circuit is None:
            return circuits
        cache = self.__dict__.setdefault("_composed", {})
        init_fp = _circuit_fingerprint(self._initial_state_circuit)
        out = []
        for circ in circuits:
            if hasattr(circ, "layers") and not hasattr(circ, "data"):  # a genome: compose needs its circuit form
                circ = circ.to_circuit() if hasattr(circ, "to_circuit") else circ.get_parameterized_quantum_circuit()
            hit = cache.get(id(circ))
            fp = (_circuit_fingerprint(circ), init_fp)  # either circuit edited in place since: compose again
            if hit is None or hit[0] is not circ or hit[2] != fp:
                if len(cache) > 1024:
                    cache.clear()
                hit = cache[id(circ)] = (circ, self._initial_state_circuit.compose(circ, inplace=False), fp)
            out.append(hit[1])
        return out


class B200OperatorCircuitEvaluator(BaseCircuitEvaluator, _WithInitialState):
    """<psi(theta)|H|psi(theta)> of every circuit, exact up to the estimator's ``precision`` noise
    (drop-in for ``OperatorCircuitEvaluator``, circuit_evaluation.py:162-219)."""

    def __init__(self, estimator: B200EstimatorV2, estimator_precision: float, operator, initial_state_circuit=None):
        if not isinstance(estimator, B200EstimatorV2):
            raise TypeError("B200OperatorCircuitEvaluator needs a B200EstimatorV2 (it carries device / dtype / seed)")
        self._estimator = estimator
        self._estimator_precision = float(estimator_precision)
        self._operator = operator
        self._n_qubits = int(operator.num_qubits)
        _check_initial_state(initial_state_circuit, self._n_qubits, "the amount of qubits in the given operator")
        self._initial_state_circuit = initial_state_circuit

    def evaluate_circuits(self, circuits: list, parameter_values: list[list[float]]) -> list[float]:
        pairs = [(c, p) for c, p in zip(self._prepend(circuits), parameter_values) if c is not None and p is not None]
        try:
            evs = self._estimator.expectation_values([c for c, _ in pairs], [p for _, p in pairs], self._operator)
        except (ValueError, TypeError):
            raise
        except Exception as exc:
            raise CircuitEvaluatorException(str(exc)) from exc
        if self._estimator_precision:
            evs = [float(self._estimator._noisy(np.asarray(e), self._estimator_precision)) for e in evs]
        return [float(e) for e in evs]

    @property
    def n_qubits(self) -> int:
        return self._n_qubits


class _SamplerEvaluator(BaseCircuitEvaluator, _WithInitialState):
    def __init__(self, sampler: B200SamplerV2, sampler_shots: Optional[int], alpha: float):
        if not isinstance(sampler, B200SamplerV2):
            raise TypeError(f"{type(self).__name__} needs a B200SamplerV2 (it carries device / dtype / seed)")
        self._sampler = sampler
        self._sampler_shots = None if sampler_shots is None else int(sampler_shots)  # None: exact values, no shots
        ex.check_alpha(alpha)
        self._alpha = float(alpha)

    def _exact(self, circuits, parameter_values, operator, kind: str) -> list[float]:
        pairs = [(c, p) for c, p in zip(self._prepend(circuits), parameter_values) if c is not None and p is not None]
        try:
            values = self._sampler._exact(kind, [c for c, _ in pairs], [p for _, p in pairs], operator, self._alpha)
        except (ValueError, TypeError, NotImplementedError):
            raise
        except Exception as exc:
            raise CircuitEvaluatorException(str(exc)) from exc
        return [float(v) for v in values]

    def _distributions(self, circuits, parameter_values):
        try:
            return measure_quasi_distributions(self._prepend(circuits), parameter_values, self._sampler, self._sampler_shots)
        except (ValueError, TypeError):
            raise
        except Exception as exc:
            raise CircuitEvaluatorException(str(exc)) from exc


class B200OperatorSamplerCircuitEvaluator(_SamplerEvaluator):
    """Shots -> distribution -> diagonal-operator expectation / CVaR(alpha)
    (drop-in for ``OperatorSamplerCircuitEvaluator``, circuit_evaluation.py:94-159)."""

    def __init__(self, sampler: B200SamplerV2, sampler_shots: int, operator, alpha: float = 1.0, initial_state_circuit=None):
        if not (hasattr(operator, "to_list") or hasattr(operator, "masks")) or not hasattr(operator, "num_qubits"):
            raise ValueError("If using a sampler to estimate the expectation value, the operator must be a SparsePauliOp!")
        super().__init__(sampler, sampler_shots, alpha)
        self._operator = operator
        n, x, z, c = operator_terms(operator)
        if np.any(x):
            raise ValueError("Operator string contains non-diagonal terms")  # [upstream] sampled_expectation_value
        self._n_qubits = n
        self._z_masks, self._coeffs = ex.merge_diagonal_terms(z, np.real(c))
        _check_initial_state(initial_state_circuit, n, "the amount of qubits in the given operator")
        self._initial_state_circuit = initial_state_circuit

    def evaluate_circuits(self, circuits: list, parameter_values: list[list[float]]) -> list[float]:
        if self._sampler_shots is None:  # exact: sum p E for alpha ~ 1 (as the sampled branch below), the sorted lower tail otherwise
            return self._exact(circuits, parameter_values, self._operator, "exp" if ex._close(self._alpha, 1) else "cvar")
        # the quasi-distributions of measure_quasi_distributions (circuit_evaluation.py:29-59) as (states, counts) arrays in
        # ascending state order -- the same entries, in the same order, as the dict route, without 10 000-entry dicts
        pairs = [(c, p) for c, p in zip(self._prepend(circuits), parameter_values) if c is not None and p is not None]
        try:
            idx = self._sampler.sample_indices([c for c, _ in pairs], [p for _, p in pairs], self._sampler_shots)
        except (ValueError, TypeError):
            raise
        except Exception as exc:
            raise CircuitEvaluatorException(str(exc)) from exc
        uniq = [np.unique(row, return_counts=True) for row in idx]
        if not uniq:
            return []
        # energies of all distinct sampled states in one device call (E(k) = sum_t c_t (-1)^{popcount(k & z_t)})
        ham = self._sampler.hamiltonian_for(self._operator, build_table=False)
        flat = self._sampler.engine.diag_energies(ham, np.concatenate([v for v, _ in uniq]).astype(np.uint64))
        out, pos = [], 0
        for states, counts in uniq:
            probs = counts / float(self._sampler_shots)
            energies = flat[pos : pos + states.size]
            pos += states.size
            if ex._close(self._alpha, 1):
                out.append(float(np.dot(probs, energies)))  # [upstream] sampled_expectation_value
            else:
                out.append(float(ex.lower_tail_expectation_arrays(probs, energies, self._alpha)))
        return out

    @property
    def n_qubits(self) -> int:
        return self._n_qubits


class B200BitstringCircuitEvaluator(_SamplerEvaluator):
    """Shots -> distribution -> user function on bitstrings -> expectation / CVaR(alpha)
    (drop-in for ``BitstringCircuitEvaluator``, circuit_evaluation.py:222-291)."""

    def __init__(self, sampler: B200SamplerV2, sampler_shots: int, bitstring_evaluator, alpha: float = 1.0, initial_state_circuit=None):
        self._bitstring_evaluator = bitstring_evaluator
        n = int(bitstring_evaluator.input_length)
        if initial_state_circuit is not None and initial_state_circuit.num_qubits != n:
            raise ValueError(
                f"The amount of qubits in the initial state circuit ({initial_state_circuit.num_qubits} "
                + f"does not match the input length of the BitstringEvaluator ({n})!"
            )
        super().__init__(sampler, sampler_shots, alpha)
        self._initial_state_circuit = initial_state_circuit
        self._diagonal_op = None
        if hasattr(bitstring_evaluator, "diagonal_terms"):
            from .operators import SparsePauliOp

            z, c = bitstring_evaluator.diagonal_terms
            self._diagonal_op = SparsePauliOp._raw(n, [0] * len(z), [int(v) for v in z], [float(v) for v in c])
        elif self._sampler_shots is None:
            raise ValueError(
                "exact evaluation (sampler_shots=None) needs a BitstringEvaluator with diagonal_terms "
                "(DiagonalEnergyBitstringEvaluator): the exact distribution would call the evaluator on all 2^n bitstrings"
            )

    def evaluate_circuits(self, circuits: list, parameter_values: list[list[float]]) -> list[float]:
        if self._sampler_shots is None:
            return self._exact(circuits, parameter_values, self._diagonal_op, "cvar")
        n = self.n_qubits
        vectorised = getattr(self._bitstring_evaluator, "evaluate_states", None)
        if vectorised is None:  # the reference contract: one call of the user's function per distinct bitstring
            return [
                float(ex.expectation_with_bitstring_evaluator(dist, self._bitstring_evaluator, self._alpha, num_bits=n))
                for dist in self._distributions(circuits, parameter_values)
            ]
        # evaluators that can value many basis states at once (DiagonalEnergyBitstringEvaluator: on the device)
        pairs = [(c, p) for c, p in zip(self._prepend(circuits), parameter_values) if c is not None and p is not None]
        try:
            idx = self._sampler.sample_indices([c for c, _ in pairs], [p for _, p in pairs], self._sampler_shots)
        except (ValueError, TypeError):
            raise
        except Exception as exc:
            raise CircuitEvaluatorException(str(exc)) from exc
        uniq = [np.unique(row, return_counts=True) for row in idx]
        if not uniq:
            return []
        states_all = np.concatenate([v for v, _ in uniq]).astype(np.uint64)
        if self._diagonal_op is not None:  # a diagonal energy: all distinct states of the population in one device call
            ham = self._sampler.hamiltonian_for(self._diagonal_op, build_table=False)
            values = self._sampler.engine.diag_energies(ham, states_all)
        else:
            values = np.asarray(vectorised(states_all), dtype=np.float64)
        out, pos = [], 0
        for states, counts in uniq:
            probs = counts / float(self._sampler_shots)
            out.append(float(ex.lower_tail_expectation_arrays(probs, values[pos : pos + states.size], self._alpha)))
            pos += states.size
        return out

    @property
    def n_qubits(self) -> int:
        return int(self._bitstring_evaluator.input_length)
