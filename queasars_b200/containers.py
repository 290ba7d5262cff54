"""Result / pub containers of the Qiskit V2 primitive contract, restricted to what the reference's
evaluators and primitive wrappers touch:

  * ``job.result()`` -> iterable + int-indexable ``PrimitiveResult`` with ``.metadata``
    (/root/reference/queasars/circuit_evaluation/mutex_primitives.py:253-260, 317-324)
  * ``pub_result.data.evs`` (circuit_evaluation.py:215) and ``pub_result.data["meas"].get_counts()`` (:55)
  * ``EstimatorPub.coerce / SamplerPub.coerce`` (mutex_primitives.py:248, 312) and the keyword
    constructor used at transpiling_primitives.py:73-79
  * ``QuasiDistribution(data, shots=)`` with integer keys and ``binary_probabilities()``
    (circuit_evaluation.py:56-59, expectation_calculation.py:96)

When real Qiskit is importable its own classes are used by callers; these are the stand-ins otherwise
and what ``B200EstimatorV2`` / ``B200SamplerV2`` return in either case (attribute-compatible).
"""
from __future__ import annotations

from abc import ABC, abstractmethod
from concurrent.futures import ThreadPoolExecutor
from typing import Any, Iterable, Mapping, Optional, Sequence

import numpy as np


class DataBin:
    def __init__(self, *, shape: tuple = (), **fields):
        object.__setattr__(self, "_fields", dict(fields))
        object.__setattr__(self, "shape", shape)

    def __getattr__(self, name):
        try:
            return self._fields[name]
        except KeyError as exc:
            raise AttributeError(name) from exc

    def __getitem__(self, key):
        return self._fields[key]

    def __contains__(self, key):
        return key in self._fields

    def keys(self):
        return self._fields.keys()

    def items(self):
        return self._fields.items()

    def __repr__(self):
        return f"DataBin({', '.join(f'{k}=...' for k in self._fields)})"


class ShotRegister:
    """Shot outcomes of one classical register (upstream ``BitArray``): basis-state indices per shot.  ``shape``: the pub's
    parameter shape; ``indices`` is then ``shape + (num_shots,)`` and ``loc`` picks one position of it (``loc=None`` pools
    every position, as upstream's ``BitArray`` does)."""

    def __init__(self, indices: np.ndarray, num_bits: int, shape: tuple = ()):
        self.shape = tuple(int(s) for s in shape)
        self._indices = np.asarray(indices, dtype=np.int64).reshape(self.shape + (-1,) if self.shape else (-1,))
        self.num_bits = int(num_bits)

    @property
    def num_shots(self) -> int:
        return int(self._indices.shape[-1])

    @property
    def indices(self) -> np.ndarray:
        return self._indices

    def _select(self, loc) -> np.ndarray:
        if loc is None:
            return self._indices.reshape(-1)
        if not self.shape:
            raise IndexError("a register of shape () has no positions to select")
        return np.asarray(self._indices[loc], dtype=np.int64).reshape(-1)

    def get_int_counts(self, loc=None) -> dict[int, int]:
        vals, cnts = np.unique(self._select(loc), return_counts=True)
        return {int(v): int(c) for v, c in zip(vals, cnts)}

    def get_counts(self, loc=None) -> dict[str, int]:
        width = self.num_bits
        return {format(v, f"0{width}b"): c for v, c in self.get_int_counts(loc).items()}

    def get_bitstrings(self, loc=None) -> list[str]:
        width = self.num_bits
        return [format(int(v), f"0{width}b") for v in self._select(loc)]


class PubResult:
    def __init__(self, data: DataBin, metadata: Optional[dict] = None):
        self.data = data
        self.metadata = metadata or {}


class SamplerPubResult(PubResult):
    def join_data(self, names=None):
        keys = list(self.data.keys()) if names is None else list(names)
        if len(keys) != 1:
            raise NotImplementedError("join_data over several registers")
        return self.data[keys[0]]


class PrimitiveResult:
    def __class_getitem__(cls, item):  # upstream is Generic[T]; annotations like PrimitiveResult[PubResult] must work
        return cls

    def __init__(self, pub_results: Iterable[PubResult], metadata: Optional[dict] = None):
        self._pub_results = list(pub_results)
        self.metadata = metadata or {}

    def __getitem__(self, index):
        return self._pub_results[index]

    def __len__(self):
        return len(self._pub_results)

    def __iter__(self):
        return iter(self._pub_results)


class BasePrimitiveJob(ABC):
    def __class_getitem__(cls, item):  # upstream is Generic[ResultT, StatusT]
        return cls

    @abstractmethod
    def result(self):
        ...

    def done(self) -> bool:
        return True

    def running(self) -> bool:
        return False

    def cancelled(self) -> bool:
        return False

    def in_final_state(self) -> bool:
        return True

    def cancel(self):
        return False

    def status(self):
        return "DONE"

    def job_id(self) -> str:
        return f"b200-{id(self):x}"


class PrimitiveJob(BasePrimitiveJob):
    """Thread-backed job like upstream ``qiskit.primitives.primitive_job.PrimitiveJob``."""

    def __init__(self, function, *args, **kwargs):
        self._function, self._args, self._kwargs = function, args, kwargs
        self._future = None

    def _submit(self):
        if self._future is not None:
            raise RuntimeError("Primitive job has been submitted already.")
        executor = ThreadPoolExecutor(max_workers=1)
        self._future = executor.submit(self._function, *self._args, **self._kwargs)
        executor.shutdown(wait=False)

    def result(self):
        if self._future is None:
            raise RuntimeError("Primitive job has not been submitted yet.")
        return self._future.result()

    def done(self) -> bool:
        return self._future is not None and self._future.done()


class FinishedJob(BasePrimitiveJob):
    """Job whose work was performed eagerly on the calling thread (no PrimitiveJob thread per run)."""

    def __init__(self, result: Any = None, error: Optional[BaseException] = None):
        self._result, self._error = result, error

    def result(self):
        if self._error is not None:
            raise self._error
        return self._result


def _as_param_array(values) -> np.ndarray:
    if values is None:
        return np.zeros((0,), dtype=np.float64)
    if isinstance(values, Mapping):
        raise TypeError("mapping-valued parameter_values need the circuit to be resolved; pass a sequence")
    return np.asarray(values, dtype=np.float64)


class EstimatorPub:
    def __init__(self, circuit, observables, parameter_values=None, precision: Optional[float] = None, validate: bool = True):
        self.circuit = circuit
        self.observables = observables
        self.parameter_values = parameter_values
        self.precision = precision

    @classmethod
    def coerce(cls, pub, precision: Optional[float] = None) -> "EstimatorPub":
        if hasattr(pub, "circuit") and hasattr(pub, "observables"):
            if getattr(pub, "precision", None) is None and precision is not None:
                return cls(pub.circuit, pub.observables, pub.parameter_values, precision, validate=False)
            return pub
        pub = tuple(pub)
        if len(pub) not in (2, 3, 4):
            raise ValueError(f"The length of pub must be 2, 3 or 4, but length {len(pub)} is given.")
        circuit, observables = pub[0], pub[1]
        values = pub[2] if len(pub) > 2 else None
        if len(pub) > 3 and pub[3] is not None:
            precision = pub[3]
        return cls(circuit, observables, values, precision)


class SamplerPub:
    def __init__(self, circuit, parameter_values=None, shots: Optional[int] = None, validate: bool = True):
        self.circuit = circuit
        self.parameter_values = parameter_values
        self.shots = shots

    @classmethod
    def coerce(cls, pub, shots: Optional[int] = None) -> "SamplerPub":
        if hasattr(pub, "circuit") and hasattr(pub, "shots"):
            if pub.shots is None and shots is not None:
                return cls(pub.circuit, pub.parameter_values, shots, validate=False)
            return pub
        if hasattr(pub, "num_qubits") and hasattr(pub, "data"):  # a bare circuit
            return cls(pub, None, shots)
        pub = tuple(pub)
        if len(pub) not in (1, 2, 3):
            raise ValueError(f"The length of pub must be 1, 2 or 3, but length {len(pub)} is given.")
        values = pub[1] if len(pub) > 1 else None
        if len(pub) > 2 and pub[2] is not None:
            shots = pub[2]
        return cls(pub[0], values, shots)


class QuasiDistribution(dict):
    """``qiskit.result.QuasiDistribution``: int-keyed dict; str keys ('0101', '0b..', '0x..') are converted."""

    def __init__(self, data: Mapping, shots: Optional[int] = None, stddev_upper_bound: Optional[float] = None):
        self.shots = shots
        self._stddev_upper_bound = stddev_upper_bound
        conv = {}
        for key, val in data.items():
            if isinstance(key, str):
                key = int(key, 0) if key[:2] in ("0x", "0b") else int(key, 2)
            conv[int(key)] = val
        super().__init__(conv)

    def binary_probabilities(self, num_bits: Optional[int] = None) -> dict[str, float]:
        n = len(bin(max(self.keys(), default=0))) - 2 if num_bits is None else num_bits
        return {format(key, "b").zfill(n): value for key, value in self.items()}

    def hex_probabilities(self) -> dict[str, float]:
        return {hex(key): value for key, value in self.items()}


class ProbDistribution(QuasiDistribution):
    pass
