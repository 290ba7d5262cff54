"""B200-native (sm_100a) circuit evaluation for QUEASARS' EVQE loop.

Public surface (mirrors /root/reference/queasars/circuit_evaluation):
  evaluators   B200OperatorCircuitEvaluator, B200OperatorSamplerCircuitEvaluator, B200BitstringCircuitEvaluator,
               measure_quasi_distributions, BitstringEvaluator
  primitives   B200EstimatorV2, B200SamplerV2 (Qiskit V2 primitive contract)
  engine       Engine (batched submission through the C-ABI in include/queasars_b200.h)
  front end    gate_list.from_circuit / from_evqe_individual, circuit.QuantumCircuit (Qiskit-API stand-in)
Importing the package never touches CUDA; the first evaluation loads the native library and fails loudly if
it has not been built or no B200 is present (there is no CPU fallback).
"""
from .bitstring_evaluation import BitstringEvaluator, BitstringEvaluatorException, DiagonalEnergyBitstringEvaluator  # noqa: F401
from .circuit import ClassicalRegister, Clbit, CU3Gate, Parameter, QuantumCircuit, circuit_to_gate  # noqa: F401
from .operators import SparsePauliOp  # noqa: F401

__all__ = [
    "BitstringEvaluator",
    "BitstringEvaluatorException",
    "DiagonalEnergyBitstringEvaluator",
    "QuantumCircuit",
    "ClassicalRegister",
    "Clbit",
    "Parameter",
    "CU3Gate",
    "circuit_to_gate",
    "SparsePauliOp",
    "Engine",
    "B200EstimatorV2",
    "B200SamplerV2",
    "B200OperatorCircuitEvaluator",
    "B200OperatorSamplerCircuitEvaluator",
    "B200BitstringCircuitEvaluator",
    "measure_quasi_distributions",
]

_LAZY = {
    "Engine": "engine",
    "B200EstimatorV2": "primitives",
    "B200SamplerV2": "primitives",
    "B200OperatorCircuitEvaluator": "evaluators",
    "B200OperatorSamplerCircuitEvaluator": "evaluators",
    "B200BitstringCircuitEvaluator": "evaluators",
    "measure_quasi_distributions": "evaluators",
    "CircuitEvaluatorException": "evaluators",
}


def __getattr__(name):
    if name in _LAZY:
        import importlib

        return getattr(importlib.import_module(f"{__name__}.{_LAZY[name]}"), name)
    raise AttributeError(name)
