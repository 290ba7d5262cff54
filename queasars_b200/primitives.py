"""B200 Estimator / Sampler primitives implementing the Qiskit V2 primitive *contract* the reference consumes

    estimator.run(pubs, *, precision=None).result()[i].data.evs          (circuit_evaluation.py:210-215)
    sampler.run(pubs, *, shots=None).result()[i].data["meas"].get_counts()  (circuit_evaluation.py:54-55)

so the unmodified reference evaluators and wrappers (``TranspilingEstimatorV2``, ``(Batching)Mutex*``,
``Configured*V2``; /root/reference/queasars/circuit_evaluation/*.py) can be handed these objects.  Pubs may
be tuples, ``EstimatorPub`` / ``SamplerPub`` objects (real Qiskit's or the stand-ins) or generators.

Semantics follow [upstream] ``StatevectorEstimator`` / ``StatevectorSampler`` (qiskit 2.4.2):
  * estimator: ``evs = Re <psi|H|psi>``; with ``precision != 0`` Gaussian noise
    ``default_rng(seed).normal(evs, precision)`` from a fresh generator per pub, ``stds = precision``
  * sampler: ``Generator.choice`` = ``cumsum(|psi|^2)`` CDF + ``searchsorted(uniforms, side='right')`` with
    ``uniforms = default_rng(seed).random(shots)``, a fresh generator per pub when ``seed`` is an int.
QUEASARS itself only sends zero-dimensional pubs (one parameter vector, one observable).  Arrays are accepted too:
  * estimator: an observables array of several elements (``ObservablesArray``, nested lists of ``SparsePauliOp``s,
    ``{label: coeff}`` dicts or labels) is broadcast against the parameter shape, ``evs.shape ==
    np.broadcast_shapes(obs_shape, param_shape)``; every distinct parameter row is simulated once and all distinct
    observables are reduced from that one state (``expectation_values_many``).  A pub with exactly one observable keeps
    the single-observable route, and ``[H]`` gives the parameter shape (upstream: ``(1,)``).
  * sampler: ``parameter_values`` of shape S give one submission over all rows and ``data.meas`` of shape S
    (``get_counts(loc=None)`` pools every position, as upstream's ``BitArray``).
"""
from __future__ import annotations

import ctypes
import threading
import weakref
from typing import Iterable, Optional, Sequence

import numpy as np

from . import _native
from . import containers as ct
from . import expectation as ex
from .batching import CoalescingQueue
from .engine import Engine, HamiltonianHandle, ObservablesHandle, PlanHandle
from .gate_list import from_circuit_or_none, from_circuit

_engines: dict = {}
_engines_lock = threading.Lock()


def get_engine(device: int = 0, dtype: str = "complex128") -> Engine:
    """Process-wide engine per (device, dtype); created lazily so configuration objects stay picklable."""
    key = (int(device), str(np.dtype(dtype).name))
    with _engines_lock:
        eng = _engines.get(key)
        if eng is None:
            eng = _engines[key] = Engine(device=device, dtype=dtype)
        return eng


def _is_genome(obj) -> bool:
    """An EVQE individual (the reference's ``EVQEIndividual`` or ``queasars_b200.genome.Individual``) handed in where a circuit
    is expected: the direct genome -> gate-list front end (SURVEY.md section 8f-3) skips the QuantumCircuit altogether."""
    return hasattr(obj, "layers") and hasattr(obj, "parameter_values") and not hasattr(obj, "data")


def _parse(circuit):
    if _is_genome(circuit):
        from .gate_list import from_evqe_individual

        return from_evqe_individual(circuit)
    return from_circuit_or_none(circuit)


def _width(circuit) -> int:
    return int(circuit.n_qubits if _is_genome(circuit) else circuit.num_qubits)


def _circuit_fingerprint(circuit) -> tuple:
    """Cheap guard against in-place edits of a circuit between two evaluations (Qiskit circuits are mutable; the reference
    re-transpiles on every call: transpiling_primitives.py:47, 73-80): instruction count and parameter count.  A circuit
    whose fingerprint changed is re-parsed and re-compiled."""
    if _is_genome(circuit):
        return (len(circuit.layers),)  # genomes are immutable value objects
    try:
        version = getattr(circuit, "_b200_version", None)  # the stand-in circuit class counts its mutations (O(1))
        if version is not None:
            return (len(circuit.data), version)
        return (len(circuit.data), int(circuit.num_parameters))  # Qiskit: both O(1)
    except Exception:
        return ()


def _operator_fingerprint(operator) -> tuple:
    """Term count + hash of the coefficients (``SparsePauliOp.coeffs`` can be assigned in place)."""
    try:
        coeffs = np.asarray(operator.coeffs if hasattr(operator, "coeffs") else operator.masks()[2])
        return (int(coeffs.size), hash(coeffs.tobytes()))
    except Exception:
        return ()


class _CircuitCache:
    """circuit object -> parsed gate list and, per device, compiled plan; keyed by identity (the optimizer loop re-submits the
    *same* circuit object on every objective call: evqe/evolutionary_algorithm/mutation.py:63-75) and guarded by a
    fingerprint so a circuit edited in place is compiled again."""

    def __init__(self, engines: Sequence[Engine]):
        self._engines = list(engines)
        self._lock = threading.Lock()
        self._by_id: dict = {}

    def _entry(self, circuit):
        key = id(circuit)
        fp = _circuit_fingerprint(circuit)
        hit = self._by_id.get(key)  # (dict.get is atomic under the GIL: the hot path takes no lock)
        if hit is not None and hit["ref"]() is circuit and hit["fp"] == fp:
            return hit
        entry = {"ref": None, "fp": fp, "gates": _parse(circuit), "plans": {}, "home": None}
        try:
            entry["ref"] = weakref.ref(circuit, lambda _r, k=key: self._by_id.pop(k, None))
        except TypeError:  # not weak-referenceable: do not cache by identity
            entry["ref"] = lambda: None
            return entry
        with self._lock:
            self._by_id[key] = entry
        return entry

    def gates_for(self, circuit):
        return self._entry(circuit)

    def plan_for(self, circuit, slot: int = 0, entry=None, probabilities_only: bool = False) -> Optional[PlanHandle]:
        """``probabilities_only``: the caller needs |psi_k|^2 only (diagonal observable / sampling), so the plan may leave the
        diagonal phases pending at the end of the circuit unapplied (engine.rewritten)."""
        entry = self._entry(circuit) if entry is None else entry
        if entry["gates"] is None:
            return None
        plan = entry["plans"].get((slot, probabilities_only))
        if plan is None:
            # identity-cached circuits are the ones an optimizer loop re-submits: worth caching their constant prefix state
            plan = self._engines[slot].compile_with_prefix_reuse(entry["gates"], drop_final_phases=probabilities_only)
            entry["plans"][(slot, probabilities_only)] = plan
        return plan

    def bound_plan(self, circuit, values, slot: int = 0, probabilities_only: bool = False) -> PlanHandle:
        """Slow path for circuits whose angles are not affine in single parameters: bind on the host."""
        bound = circuit.assign_parameters(list(values)) if len(values) else circuit
        return self._engines[slot].compile(from_circuit(bound), drop_final_phases=probabilities_only)


def _rotate_for_process(devices: list) -> list:
    """Device order for this process.  A primitive pickled into worker processes (the reference's dask route: evqe.py:38-44,
    mutation.py:194-218) keeps its device SET but every process starts filling it at a different device, so single-circuit
    calls from different workers do not all land on the first GPU."""
    if len(devices) < 2:
        return devices
    import os

    k = os.getpid() % len(devices)
    return devices[k:] + devices[:k]


class _B200Primitive:
    """Shared runtime of the two primitives.  ``devices``: the GPUs this primitive may use -- a list of CUDA device indices
    or "all" (every device visible to the process); default: the single ``device``.  One native engine per device, one
    worker thread per device; every submitted list is split over the devices by estimated cost (sweeps x state size),
    plans and Hamiltonians are replicated lazily, results come back in submission order.  This is the reference's
    population parallelism (ThreadPoolExecutor / dask workers around ONE primitive: evqe.py:232-236, selection.py:75-82)
    mapped onto several GPUs behind the unchanged evaluator interface; the evaluations are independent, so there is no
    collective."""

    def __init__(self, device: int = 0, dtype: str = "complex128", seed=None, coalesce: bool = True, devices=None, shard_min_qubits: Optional[int] = None):
        self.device, self.dtype, self.seed, self.coalesce = int(device), str(np.dtype(dtype).name), seed, bool(coalesce)
        # circuits of at least this many qubits are evaluated as ONE statevector sharded over the device set (sharded.py);
        # None = as soon as the state does not fit one device's workspace (34 qubits complex128 on a 180 GB B200)
        self.shard_min_qubits = None if shard_min_qubits is None else int(shard_min_qubits)
        if devices is not None and devices != "all":
            devices = [int(d) for d in devices]
            if not devices or len(set(devices)) != len(devices):
                raise ValueError("devices must be a non-empty list of distinct CUDA device indices, or 'all'")
        self.devices = devices
        self._origin_pid = None
        self._init_runtime()

    def _init_runtime(self):
        self._engines_obj: Optional[list] = None
        self._cache_obj: Optional[_CircuitCache] = None
        self._ham_cache: dict = {}
        self._queue_obj: Optional[CoalescingQueue] = None
        self._pool_obj = None
        self._sharded_obj: dict = {}
        self._shard_lock = threading.Lock()  # ONE sharded state per primitive: wide circuits are evaluated one at a time
        self._lock = threading.Lock()
        self._rr = 0  # round-robin start of the device choice for small submissions
        self._last_resolution = None  # (probabilities_only, cache entries, device slots, plans) of the previous submission

    # picklable: CUDA handles are per process and re-created lazily (the dask route of the reference pickles
    # evaluators + primitives into worker processes: evqe.py:38-44)
    def __getstate__(self):
        import os

        return {"device": self.device, "dtype": self.dtype, "seed": self.seed, "coalesce": self.coalesce, "devices": self.devices,
                "shard_min_qubits": self.shard_min_qubits, "_origin_pid": self._origin_pid or os.getpid()}

    def __setstate__(self, state):
        self.__dict__.update(state)
        self._init_runtime()

    def _device_list(self) -> list:
        import os

        if self.devices is None:
            return [self.device]
        devices = list(range(_native.device_count())) if self.devices == "all" else list(self.devices)
        if not devices:
            raise RuntimeError("no CUDA device visible (queasars_b200 has no CPU fallback)")
        # un-pickled in another process than the one that configured it: start at a process-specific device
        return _rotate_for_process(devices) if self._origin_pid not in (None, os.getpid()) else devices

    @property
    def engines(self) -> list:
        with self._lock:
            if self._engines_obj is None:
                self._engines_obj = [get_engine(d, self.dtype) for d in self._device_list()]
            return self._engines_obj

    @property
    def engine(self) -> Engine:
        return self.engines[0]

    @property
    def _cache(self) -> _CircuitCache:
        engines = self.engines
        with self._lock:
            if self._cache_obj is None:
                self._cache_obj = _CircuitCache(engines)
            return self._cache_obj

    @property
    def _queue(self) -> CoalescingQueue:
        with self._lock:
            if self._queue_obj is None:
                self._queue_obj = CoalescingQueue(self._execute)
            return self._queue_obj

    @property
    def _pool(self):
        from concurrent.futures import ThreadPoolExecutor

        engines = self.engines
        with self._lock:
            if self._pool_obj is None:
                self._pool_obj = ThreadPoolExecutor(max_workers=len(engines), thread_name_prefix="qb-device")
            return self._pool_obj

    def hamiltonian_for(self, operator, build_table=None, slot: int = 0, fingerprint=None) -> HamiltonianHandle:
        key = (id(operator), build_table, slot)
        fp = _operator_fingerprint(operator) if fingerprint is None else fingerprint
        with self._lock:
            hit = self._ham_cache.get(key)
            if hit is not None and hit[0] is operator and hit[2] == fp:
                return hit[1]
        engines = self.engines  # (takes the lock itself: not inside the block below)
        handle = engines[slot].hamiltonian(operator, build_table=build_table)
        with self._lock:
            if len(self._ham_cache) > 64 * len(engines):
                self._ham_cache.clear()
            self._ham_cache[key] = (operator, handle, fp)
        return handle

    def observables_for(self, operators: Sequence, slot: int = 0, fingerprints=None) -> ObservablesHandle:
        """Device form of a set of observables on device ``slot``, cached like ``hamiltonian_for``: by the operators' identities,
        guarded by their fingerprints against in-place edits."""
        operators = tuple(operators)
        key = ("obs", tuple(id(op) for op in operators), slot)
        fps = tuple(_operator_fingerprint(op) for op in operators) if fingerprints is None else tuple(fingerprints)
        with self._lock:
            hit = self._ham_cache.get(key)
            if hit is not None and len(hit[0]) == len(operators) and all(a is b for a, b in zip(hit[0], operators)) and hit[2] == fps:
                return hit[1]
        engines = self.engines
        handle = engines[slot].observables(operators)
        with self._lock:
            if len(self._ham_cache) > 64 * len(engines):
                self._ham_cache.clear()
            self._ham_cache[key] = (operators, handle, fps)
        return handle

    # ------------------------------------------------------------------ splitting a submission over the devices
    def _assign(self, entries: Sequence, costs: Sequence[float]) -> list:
        """entries[i] = cache entry of circuit i (or None) -> device slot per entry.  Greedy longest-processing-time over
        circuits (all rows of one circuit object stay together unless that circuit alone is more than a device's share,
        then its rows are dealt out), preferring the device that already holds the circuit's plan / cached prefix state
        while that does not unbalance the split."""
        n_dev = len(self.engines)
        if n_dev == 1:
            return [0] * len(entries)
        groups: dict = {}
        for i, en in enumerate(entries):
            groups.setdefault(id(en) if en is not None else ("row", i), []).append(i)
        total = float(sum(costs)) or 1.0
        share = total / n_dev
        units = []  # (cost, rows, home)
        for rows in groups.values():
            en = entries[rows[0]]
            home = en["home"] if en is not None else None
            cost = sum(costs[i] for i in rows)
            if cost > 1.25 * share and len(rows) > 1:  # one circuit, many parameter vectors: deal the rows out
                per = max(1, int(len(rows) * share / cost))
                for lo in range(0, len(rows), per):
                    part = rows[lo : lo + per]
                    units.append((sum(costs[i] for i in part), part, None))
            else:
                units.append((cost, rows, home))
        units.sort(key=lambda u: -u[0])
        load = [0.0] * n_dev
        out = [0] * len(entries)
        with self._lock:
            start = self._rr
            self._rr = (self._rr + 1) % n_dev
        for cost, rows, home in units:
            best = min(range(n_dev), key=lambda d: (load[d], (d - start) % n_dev))
            if home is not None and load[home] <= load[best] + 0.5 * cost:
                best = home
            load[best] += cost
            for i in rows:
                out[i] = best
                if entries[i] is not None and entries[i]["home"] is None:
                    entries[i]["home"] = best
        return out

    def _resolve_all(self, circuits, parameter_values, probabilities_only: bool = False):
        """-> list of (slot, plan, values) in submission order."""
        cache = self._cache
        # the same circuit objects in the same order as last time (an optimizer loop, a bench step): reuse the device split and
        # the plans after checking that every object is still the one that was cached and was not edited in place
        memo = self._last_resolution
        if memo is not None and len(memo[1]) == len(circuits) and memo[0] == probabilities_only:
            entries, slots, plans = memo[1], memo[2], memo[3]
            if all(en["ref"]() is c and en["fp"] == _circuit_fingerprint(c) for en, c in zip(entries, circuits)):
                return [(slot, plan, values if values is not None else ()) for slot, plan, values in zip(slots, plans, parameter_values)]
        entries = [cache.gates_for(c) for c in circuits]
        costs = []
        for en in entries:
            gates = en["gates"]
            costs.append(float(max(1, len(gates.ops))) if gates is not None else 1.0)
        slots = self._assign(entries, costs)
        out = []
        for circuit, values, en, slot in zip(circuits, parameter_values, entries, slots):
            plan = cache.plan_for(circuit, slot, en, probabilities_only)
            if plan is None:
                values = np.asarray(values if values is not None else (), dtype=np.float64).reshape(-1)
                out.append((slot, cache.bound_plan(circuit, values, slot, probabilities_only), np.zeros(0)))
            else:
                # the float64 conversion happens chunk by chunk inside the engine's pipelined submission, overlapped with
                # the GPU work of the previous chunk
                out.append((slot, plan, values if values is not None else ()))
        if all(en["gates"] is not None and en["ref"]() is not None for en in entries):  # (host-bound circuits are resolved per call)
            self._last_resolution = (probabilities_only, entries, slots, [o[1] for o in out])
        return out

    def _run_per_device(self, resolved, call):
        """Group ``resolved`` = [(slot, plan, values)] by device, run ``call(slot, plans, params)`` on every device's own
        worker thread, return the per-entry results in submission order."""
        by_slot: dict = {}
        for i, (slot, _, _) in enumerate(resolved):
            by_slot.setdefault(slot, []).append(i)
        results = [None] * len(resolved)

        def work(slot, rows):
            return call(slot, [resolved[i][1] for i in rows], [resolved[i][2] for i in rows])

        if len(by_slot) == 1:
            ((slot, rows),) = by_slot.items()
            for i, r in zip(rows, work(slot, rows)):
                results[i] = r
            return results
        futures = {slot: self._pool.submit(work, slot, rows) for slot, rows in by_slot.items()}
        error = None
        for slot, fut in futures.items():
            try:
                for i, r in zip(by_slot[slot], fut.result()):
                    results[i] = r
            except BaseException as exc:  # wait for every device before surfacing the first failure
                error = error or exc
        if error is not None:
            raise error
        return results

    def devices_used(self) -> list:
        return [e.device for e in self.engines]

    # ------------------------------------------------------------------ circuits too wide for one GPU
    def _needs_sharding(self, n_qubits: int) -> bool:
        if self.shard_min_qubits is not None:
            return n_qubits >= self.shard_min_qubits
        amp = 16 if self.dtype == "complex128" else 8
        return (amp << n_qubits) > self.engine.workspace_bytes

    def _sharded_state(self, n_qubits: int):
        """One state of ``n_qubits`` sharded over the largest power-of-two prefix of the device set (kept between calls: two
        shard-sized buffers per GPU).  BASELINE config C5: 35 qubits over 8 GPUs."""
        from .sharded import LocalShardedStatevector

        if self.dtype != "complex128":
            raise NotImplementedError("sharded statevectors are complex128")
        with self._lock:
            sv = self._sharded_obj.get(n_qubits)
        if sv is not None:
            return sv
        engines = self.engines
        count = 1 << int(np.log2(len(engines)))
        if count < 2 and self.shard_min_qubits is None:
            raise ValueError(
                f"a {n_qubits}-qubit statevector does not fit one GPU ({self.engine.workspace_bytes >> 30} GiB workspace): "
                "give the primitive a device set (devices=[...] or 'all') to shard it"
            )
        with self._lock:
            for old in self._sharded_obj.values():  # one resident sharded state at a time: they are sized for most of the memory
                old.close()
            self._sharded_obj.clear()
        sv = LocalShardedStatevector(n_qubits, engines[:count], min_local=min(12, n_qubits - int(np.log2(count))))
        with self._lock:
            self._sharded_obj[n_qubits] = sv
        return sv

    def _bound_gates(self, circuit, values):
        """(gate list, parameter values) of one evaluation for the sharded route."""
        entry = self._cache.gates_for(circuit)
        values = np.asarray(values if values is not None else (), dtype=np.float64).reshape(-1)
        if entry["gates"] is not None:
            if values.size != entry["gates"].n_params:
                raise ValueError(f"circuit has {entry['gates'].n_params} parameters but {values.size} values were given")
            return entry["gates"], values
        bound = circuit.assign_parameters(list(values)) if len(values) else circuit
        return from_circuit(bound), np.zeros(0)

    def _submit(self, key, payload):
        if self.coalesce:
            return self._queue.submit(key, payload)
        return self._execute(key, [payload])[0]

    def _execute(self, key, payloads):
        """Evaluate the payloads (target, circuits, parameter vectors) coalesced under ``key`` as one list: circuit after circuit on
        one statevector sharded over the device set when they are too wide for one GPU, otherwise split over the devices.  Returns
        every payload's rows, stacked, in its own order."""
        circuits, values, sizes = [], [], []
        for _, circs, vals in payloads:
            sizes.append(len(circs))
            circuits.extend(circs)
            values.extend(vals)
        width, on_state, on_devices, stack = self._parts(key, payloads[0][0])
        if self._needs_sharding(width):
            flat = []
            with self._shard_lock:
                sv = self._sharded_state(width)
                for circuit, vals in zip(circuits, values):
                    gates, bound = self._bound_gates(circuit, vals)
                    sv.reset()
                    sv.run(gates, bound)
                    flat.append(on_state(sv))
        else:
            flat = on_devices(circuits, values)
        out, pos = [], 0
        for n in sizes:
            out.append(stack(flat[pos : pos + n]))
            pos += n
        return out

    def _parts(self, key, target):  # pragma: no cover - overridden
        """What ``_execute`` needs of one kind of submission: (qubit count, ``on_state(sv)`` -> the row of the sharded state just run,
        ``on_devices(circuits, values)`` -> their rows in submission order, ``stack(rows)`` -> one payload's result)."""
        raise NotImplementedError


def _float_rows(rows) -> np.ndarray:
    return np.asarray(rows, dtype=np.float64)


def _param_rows(values) -> tuple[np.ndarray, tuple]:
    """pub parameter_values -> (2-D array rows x n_params, result shape)."""
    if values is None:
        return np.zeros((1, 0)), ()
    if hasattr(values, "as_array"):  # qiskit BindingsArray
        values = values.as_array()
    arr = np.asarray(values, dtype=np.float64)
    if arr.ndim <= 1:
        return arr.reshape(1, -1), ()
    return arr.reshape(-1, arr.shape[-1]), arr.shape[:-1]


class B200EstimatorV2(_B200Primitive):
    """EstimatorV2-contract primitive backed by the CUDA statevector engine."""

    def __init__(self, device: int = 0, dtype: str = "complex128", seed=None, default_precision: float = 0.0, coalesce: bool = True, devices=None,
                 shard_min_qubits: Optional[int] = None):
        super().__init__(device, dtype, seed, coalesce, devices, shard_min_qubits)
        self.default_precision = default_precision

    def __getstate__(self):
        return {**super().__getstate__(), "default_precision": self.default_precision}

    def expectation_values(self, circuits, parameter_values, operator) -> np.ndarray:
        """Fast path used by ``B200OperatorCircuitEvaluator``: exact <H> of (circuit_i, params_i)."""
        circuits, parameter_values = list(circuits), list(parameter_values)
        if len(circuits) != len(parameter_values):
            raise ValueError(f"{len(circuits)} circuits but {len(parameter_values)} parameter vectors")
        if not circuits:
            return np.zeros(0)
        fp = _operator_fingerprint(operator)  # once per call: guards the cached device Hamiltonian against in-place edits
        sharded = self._needs_sharding(int(operator.num_qubits))
        if not sharded:
            ham = self.hamiltonian_for(operator, fingerprint=fp)  # validates the operator (and builds its device form) before anything is queued
            engines = self._engines_obj  # (built by the calls above)
            if not self.coalesce and len(engines) == 1:
                # one device, nothing to merge with other threads' requests (the optimizer loop's sequential calls): straight to the engine
                resolved = self._resolve_all(circuits, parameter_values, probabilities_only=ham.diagonal)
                return np.asarray(engines[0].expectation([r[1] for r in resolved], [r[2] for r in resolved], ham), dtype=np.float64)
        return np.asarray(self._submit(("exp", id(operator), fp), (operator, circuits, parameter_values)))

    def expectation_values_many(self, circuits, parameter_values, observables) -> np.ndarray:
        """Exact <H_j> of every (circuit_i, params_i) and every observable H_j: float64 array [len(circuits), len(observables)].
        Each circuit is simulated once and every distinct Pauli string of the set is reduced once per state."""
        circuits, parameter_values, observables = list(circuits), list(parameter_values), list(observables)
        if len(circuits) != len(parameter_values):
            raise ValueError(f"{len(circuits)} circuits but {len(parameter_values)} parameter vectors")
        if not observables:
            raise ValueError("at least one observable is needed")
        widths = {int(op.num_qubits) for op in observables}
        if len(widths) != 1:
            raise ValueError("all observables of one set must act on the same number of qubits")
        width = widths.pop()
        for c in circuits:
            if _width(c) != width:
                raise ValueError(f"a circuit acts on {_width(c)} qubits, the observables on {width}")
        if not circuits:
            return np.zeros((0, len(observables)))
        fps = tuple(_operator_fingerprint(op) for op in observables)
        if not self._needs_sharding(width):
            self.observables_for(observables, fingerprints=fps)  # validates the set (and builds its device form) before anything is queued
        key = ("many", tuple(id(op) for op in observables), fps)
        return np.asarray(self._submit(key, (observables, circuits, parameter_values)), dtype=np.float64).reshape(len(circuits), len(observables))

    def _parts(self, key, target):
        if key[0] == "many":  # target: the observables, every one evaluated on each state
            observables, fps = target, key[2]

            def many_on_devices(circuits, values):
                diagonal = self.observables_for(observables, fingerprints=fps).diagonal
                resolved = self._resolve_all(circuits, values, probabilities_only=diagonal)
                return self._run_per_device(
                    resolved, lambda slot, plans, params: list(self.engines[slot].expectation_many(plans, params, self.observables_for(observables, slot, fps)))
                )

            return (int(observables[0].num_qubits), lambda sv: np.asarray([sv.expectation(op) for op in observables], dtype=np.float64), many_on_devices,
                    lambda rows: np.asarray(rows, dtype=np.float64).reshape(len(rows), len(observables)))
        operator, fp = target, key[2]

        def on_devices(circuits, values):
            resolved = self._resolve_all(circuits, values, probabilities_only=self.hamiltonian_for(operator, fingerprint=fp).diagonal)
            return self._expectation_on_devices(resolved, operator, fp)

        return int(operator.num_qubits), lambda sv: sv.expectation(operator), on_devices, _float_rows

    def _expectation_on_devices(self, resolved, operator, fp) -> list:
        """<H> of every resolved (slot, plan, values) entry, in submission order.  One device: one blocking native call.  Several
        devices: the shares are packed here and handed to ONE native call that evaluates every device's share on that context's
        own host thread, so the GPUs are fed concurrently without per-device Python threads."""
        by_slot: dict = {}
        for i, (slot, _, _) in enumerate(resolved):
            by_slot.setdefault(slot, []).append(i)
        if len(by_slot) == 1:
            return self._run_per_device(
                resolved, lambda slot, plans, params: self.engines[slot].expectation(plans, params, self.hamiltonian_for(operator, slot=slot, fingerprint=fp))
            )
        results = [None] * len(resolved)
        shares = []
        for slot, rows in sorted(by_slot.items()):
            engine = self.engines[slot]
            ids, flat, offsets = Engine._pack([resolved[i][1] for i in rows], [resolved[i][2] for i in rows])
            shares.append((engine, rows, ids, flat, offsets, np.empty(len(rows), dtype=np.float64), self.hamiltonian_for(operator, slot=slot, fingerprint=fp)))
        if not all(hasattr(sh[0], "_ctx") for sh in shares):  # (test doubles without a native context: one blocking call per device)
            for engine, rows, *_rest, ham in shares:
                for i, r in zip(rows, engine.expectation([resolved[i][1] for i in rows], [resolved[i][2] for i in rows], ham)):
                    results[i] = r
            return results
        n = len(shares)
        lib = shares[0][0]._lib
        ctxs = (ctypes.c_void_p * n)(*[sh[0]._ctx.value for sh in shares])
        batches = (ctypes.c_int * n)(*[len(sh[1]) for sh in shares])
        ids_p = (ctypes.c_void_p * n)(*[sh[2].ctypes.data for sh in shares])
        vals_p = (ctypes.c_void_p * n)(*[sh[3].ctypes.data for sh in shares])
        offs_p = (ctypes.c_void_p * n)(*[sh[4].ctypes.data for sh in shares])
        outs_p = (ctypes.c_void_p * n)(*[sh[5].ctypes.data for sh in shares])
        hams = (ctypes.c_int64 * n)(*[sh[6].ham_id for sh in shares])
        # ONE native call: every context evaluates its share on its own host thread (qb_evaluate_expectation_multi), outside the
        # interpreter lock.  A context serves one such call at a time: the engines' submit locks are taken in device order.
        locks = [sh[0]._submit_lock for sh in sorted(shares, key=lambda sh: sh[0].device)]
        for lock in locks:
            lock.acquire()
        try:
            _native.check(lib.qb_evaluate_expectation_multi(n, ctxs, batches, ids_p, vals_p, offs_p, hams, outs_p))
        finally:
            for lock in reversed(locks):
                lock.release()
        for _, rows, _ids, _flat, _offs, out, _ham in shares:
            for i, r in zip(rows, out):
                results[i] = r
        return results

    def _noisy(self, evs: np.ndarray, precision: float) -> np.ndarray:
        if not precision:
            return evs
        rng = np.random.default_rng(self.seed)  # fresh generator per pub, like upstream
        return rng.normal(evs, precision)

    def run(self, pubs: Iterable, *, precision: Optional[float] = None):
        try:
            coerced = [ct.EstimatorPub.coerce(pub, precision) for pub in pubs]
            results = []
            for pub in coerced:
                prec = pub.precision if pub.precision is not None else self.default_precision
                rows, shape = _param_rows(pub.parameter_values)
                try:
                    ops, obs_shape = _observables_array(pub.observables)
                except TypeError:  # not an observables array this module reads: the single-observable route decides
                    ops, obs_shape = [None], ()
                if len(ops) != 1:
                    evs = self._many_evs(pub.circuit, rows, shape, ops, obs_shape)
                    evs = self._noisy(evs, float(prec or 0.0))
                    shape = evs.shape
                    results.append(
                        ct.PubResult(ct.DataBin(evs=evs, stds=np.full(shape, float(prec or 0.0)), shape=shape),
                                     metadata={"target_precision": prec, "circuit_metadata": {}})
                    )
                    continue
                evs = self.expectation_values([pub.circuit] * len(rows), list(rows), _single_observable(pub.observables))
                evs = self._noisy(np.asarray(evs, dtype=np.float64), float(prec or 0.0)).reshape(shape)
                stds = np.full(shape, float(prec or 0.0))
                results.append(
                    ct.PubResult(ct.DataBin(evs=evs, stds=stds, shape=shape), metadata={"target_precision": prec, "circuit_metadata": {}})
                )
            return ct.FinishedJob(ct.PrimitiveResult(results, metadata={"version": 2, "backend": "queasars_b200"}))
        except Exception as exc:  # surfaced by job.result(), like a PrimitiveJob would
            return ct.FinishedJob(error=exc)

    def _many_evs(self, circuit, rows: np.ndarray, param_shape: tuple, ops: list, obs_shape: tuple) -> np.ndarray:
        """evs of a pub with several observables: V2 broadcasting of the observable shape against the parameter shape; every
        distinct parameter row is simulated once and evaluated with all distinct observables in one call."""
        shape = np.broadcast_shapes(obs_shape, param_shape)  # (ValueError for shapes that do not broadcast)
        width = _width(circuit)
        for op in ops:
            if int(op.num_qubits) != width:
                raise ValueError(f"an observable acts on {int(op.num_qubits)} qubits, the circuit on {width}")
        uniq_rows, row_of = np.unique(rows, axis=0, return_inverse=True) if len(rows) > 1 else (rows, np.zeros(len(rows), dtype=np.int64))
        row_of = np.asarray(row_of).reshape(-1)
        keys, distinct, op_of = {}, [], []
        for op in ops:
            x, z, c = _op_masks(op)
            k = (x.tobytes(), z.tobytes(), c.tobytes())
            if k not in keys:
                keys[k] = len(distinct)
                distinct.append(op)
            op_of.append(keys[k])
        vals = self.expectation_values_many([circuit] * len(uniq_rows), list(uniq_rows), distinct)
        p_idx = np.broadcast_to(row_of.reshape(param_shape), shape)
        o_idx = np.broadcast_to(np.asarray(op_of, dtype=np.int64).reshape(obs_shape), shape)
        return np.asarray(vals[p_idx, o_idx], dtype=np.float64)


def _op_masks(op):
    from .engine import operator_terms

    _, x, z, c = operator_terms(op)
    return np.asarray(x, dtype=np.uint64), np.asarray(z, dtype=np.uint64), np.asarray(c, dtype=complex)


def _as_operator(obs):
    """One element of an observables array: a ``SparsePauliOp``(-like), a ``{label: coeff}`` dict or a Pauli label."""
    from .operators import SparsePauliOp

    if isinstance(obs, dict):
        if not obs:
            raise ValueError("an observable given as a dict needs at least one term")
        return SparsePauliOp.from_list(list(obs.items()))
    if isinstance(obs, str):
        return SparsePauliOp(obs)
    if hasattr(obs, "num_qubits") and (hasattr(obs, "to_list") or hasattr(obs, "masks")):
        return obs
    raise TypeError(f"cannot interpret {type(obs).__name__} as an observable")


def _observables_array(observables) -> tuple[list, tuple]:
    """A pub's observables -> (operators in row-major order, shape).  Accepts qiskit's ``ObservablesArray`` (``tolist()`` gives
    ``{label: coeff}`` dicts), nested lists / tuples, dicts, ``SparsePauliOp``s and Pauli labels."""
    obs = observables
    if hasattr(obs, "tolist") and not hasattr(obs, "to_list"):  # ObservablesArray / object ndarray
        obs = obs.tolist()
    if not isinstance(obs, (list, tuple)):
        return [_as_operator(obs)], ()
    if not obs:
        raise ValueError("an observables array needs at least one observable")
    parts = [_observables_array(o) for o in obs]
    inner = parts[0][1]
    if any(p[1] != inner for p in parts):
        raise ValueError("observables array is ragged: its nested lists differ in shape")
    return [op for p in parts for op in p[0]], (len(obs),) + inner


def _single_observable(observables):
    """QUEASARS always passes one operator per pub; unwrap qiskit's ObservablesArray / dict form."""
    obs = observables
    if hasattr(obs, "tolist") and not hasattr(obs, "to_list"):  # ObservablesArray
        obs = obs.tolist()
    if isinstance(obs, (list, tuple)):
        if len(obs) != 1:
            raise NotImplementedError("B200EstimatorV2 supports one observable per pub")
        obs = obs[0]
    if isinstance(obs, dict):  # {pauli label: coeff}
        from .operators import SparsePauliOp

        return SparsePauliOp.from_list(list(obs.items()))
    return obs


def _check_measure_all(circuit) -> None:
    """The sampler returns ONE full-width register named "meas" -- what ``measure_all`` produces and the only shape QUEASARS
    consumes (circuit_evaluation.py:50-55).  Circuits with other classical registers would get a silently different result
    from upstream's per-register BitArrays, so they are rejected."""
    cregs = getattr(circuit, "cregs", None)
    if not cregs:
        return
    if len(cregs) != 1 or getattr(cregs[0], "name", "meas") != "meas" or len(cregs[0]) != int(circuit.num_qubits):
        raise NotImplementedError("B200SamplerV2 supports circuits measured with measure_all() only (one register 'meas' over all qubits)")


class B200SamplerV2(_B200Primitive):
    """SamplerV2-contract primitive: shots drawn on the GPU from the exact statevector distribution."""

    def __init__(self, device: int = 0, dtype: str = "complex128", seed=None, default_shots: int = 1024, coalesce: bool = True, devices=None,
                 shard_min_qubits: Optional[int] = None):
        super().__init__(device, dtype, seed, coalesce, devices, shard_min_qubits)
        self.default_shots = default_shots

    def __getstate__(self):
        return {**super().__getstate__(), "default_shots": self.default_shots}

    def sample_indices(self, circuits, parameter_values, shots: int) -> np.ndarray:
        """Fast path used by the B200 sampler evaluators: int64 array [len(circuits), shots] of basis states."""
        circuits, parameter_values = list(circuits), list(parameter_values)
        if len(circuits) != len(parameter_values):
            raise ValueError(f"{len(circuits)} circuits but {len(parameter_values)} parameter vectors")
        if not circuits:
            return np.zeros((0, int(shots)), dtype=np.int64)
        # circuits of different widths must not be merged into one native batch: the width is part of the coalescing key
        widths = {_width(c) for c in circuits}
        if len(widths) != 1:
            raise ValueError("all circuits of one sampler submission must act on the same number of qubits")
        return np.asarray(self._submit(("smp", int(shots), widths.pop()), (None, circuits, parameter_values)))

    def cvar_values(self, circuits, parameter_values, operator, alpha: float) -> np.ndarray:
        """Exact (shot-free) CVaR(alpha) of the diagonal ``operator`` on every circuit's full distribution |psi|^2:
        ``expectation.lower_tail_expectation_arrays(|psi|^2, E, alpha)`` over all 2^n basis states, computed on the device
        (fast path of the sampler evaluators with ``sampler_shots=None``).  float64 array [len(circuits)].

        Circuits too wide for one GPU run as one statevector sharded over the device set, one at a time, and the CVaR comes from
        the sort-free weighted select of ``sharded._ShardedLogic.cvar`` (same definition, same stop entry, ties in logical basis
        order); that route needs at least two devices and raises ``NotImplementedError`` on one."""
        return self._exact("cvar", circuits, parameter_values, operator, float(alpha))

    def _exact(self, kind: str, circuits, parameter_values, operator, alpha: float) -> np.ndarray:
        """``kind`` "cvar": ``Engine.cvar``; "exp": sum_k |psi_k|^2 E(k) through ``Engine.expectation`` (the fused diagonal
        expectation of the last sweep)."""
        circuits, parameter_values = list(circuits), list(parameter_values)
        if len(circuits) != len(parameter_values):
            raise ValueError(f"{len(circuits)} circuits but {len(parameter_values)} parameter vectors")
        ex.check_alpha(alpha)
        if not circuits:
            return np.zeros(0)
        widths = {_width(c) for c in circuits}
        if len(widths) != 1:
            raise ValueError("all circuits of one sampler submission must act on the same number of qubits")
        width = widths.pop()
        if width != int(operator.num_qubits):
            raise ValueError(f"the circuits act on {width} qubits, the operator on {int(operator.num_qubits)}")
        fp = _operator_fingerprint(operator)
        sharded = self._needs_sharding(width)
        if not self.hamiltonian_for(operator, build_table=(False if kind == "cvar" or sharded else None), fingerprint=fp).diagonal:
            raise ValueError("Operator string contains non-diagonal terms")
        if sharded and len(self.engines) < 2:
            raise NotImplementedError(
                f"exact CVaR / expectation values of a {width}-qubit state that must be sharded need a device set of at least two GPUs "
                "(devices=[...] or 'all'); on one device use shots"
            )
        return np.asarray(self._submit((kind, id(operator), fp, alpha, width), (operator, circuits, parameter_values)), dtype=np.float64)

    def _parts(self, key, target):
        if key[0] == "smp":
            _, shots, width = key

            def sample_on_state(sv):
                rng = self.seed if isinstance(self.seed, np.random.Generator) else np.random.default_rng(self.seed)
                return sv.sample(shots, uniforms=rng.random(shots))

            def sample_on_devices(circuits, values):
                resolved = self._resolve_all(circuits, values, probabilities_only=True)
                # a fresh default_rng(seed) per pub when seed is an int (or None); a shared Generator is consumed in submission order
                if isinstance(self.seed, np.random.Generator):
                    uniforms = np.stack([self.seed.random(shots) for _ in resolved])
                else:
                    one = np.random.default_rng(self.seed).random(shots) if self.seed is not None else None
                    uniforms = np.stack([one if one is not None else np.random.default_rng().random(shots) for _ in resolved])
                rows_of: dict = {}
                for i, (slot, _, _) in enumerate(resolved):
                    rows_of.setdefault(slot, []).append(i)
                return self._run_per_device(
                    resolved, lambda slot, plans, params: list(self.engines[slot].sample(plans, params, shots, uniforms[rows_of[slot]]))
                )

            return width, sample_on_state, sample_on_devices, np.stack
        kind, _, fp, alpha, width = key
        operator = target

        def on_state(sv):
            # the select passes of _ShardedLogic.cvar, or <H> for alpha ~ 1 on the operator evaluator; the duplicate-merged terms of
            # the device Hamiltonian
            ham = self.hamiltonian_for(operator, build_table=False, fingerprint=fp)
            return sv.cvar(ham.z_masks, ham.coeffs, alpha)[0] if kind == "cvar" else sv.diagonal_expectation(ham.z_masks, ham.coeffs)

        def on_devices(circuits, values):
            def call(slot, plans, params):
                engine = self.engines[slot]
                if kind == "cvar":
                    return list(engine.cvar(plans, params, self.hamiltonian_for(operator, build_table=False, slot=slot, fingerprint=fp), alpha))
                return list(engine.expectation(plans, params, self.hamiltonian_for(operator, slot=slot, fingerprint=fp)))

            return self._run_per_device(self._resolve_all(circuits, values, probabilities_only=True), call)

        return width, on_state, on_devices, _float_rows

    def run(self, pubs: Iterable, *, shots: Optional[int] = None):
        try:
            coerced = [ct.SamplerPub.coerce(pub, shots) for pub in pubs]
            results = []
            for pub in coerced:
                n_shots = int(pub.shots if pub.shots is not None else self.default_shots)
                rows, shape = _param_rows(pub.parameter_values)
                _check_measure_all(pub.circuit)
                if shape == ():
                    idx = self.sample_indices([pub.circuit], [rows[0]], n_shots)[0]
                else:  # a parameter array: one submission over all rows, one register position per row
                    idx = self.sample_indices([pub.circuit] * len(rows), list(rows), n_shots).reshape(shape + (n_shots,))
                reg = ct.ShotRegister(idx, int(pub.circuit.num_qubits), shape)
                results.append(ct.SamplerPubResult(ct.DataBin(meas=reg, shape=shape), metadata={"shots": n_shots, "circuit_metadata": {}}))
            return ct.FinishedJob(ct.PrimitiveResult(results, metadata={"version": 2, "backend": "queasars_b200"}))
        except Exception as exc:
            return ct.FinishedJob(error=exc)
