"""Python face of the native engine: compiles gate lists into device plans, uploads Hamiltonians and
submits *batches* of (plan, parameter vector) evaluations through the C-ABI.

This is the "batched submission of each generation's circuits" named by the north star: where the
reference funnels concurrent threads' pubs through ``BatchingMutexPrimitiveJobRunner`` with a fixed 0.1 s
sleep (/root/reference/queasars/circuit_evaluation/mutex_primitives.py:67-199), one ``Engine.expectation``
/ ``Engine.sample`` call evaluates the whole list in one native call; ``queasars_b200.batching`` adds the
cross-thread coalescing on top.
"""
from __future__ import annotations

import ctypes
import functools
import math
import os
import threading
import weakref
from ctypes import byref, c_double, c_int64, c_void_p
from typing import Optional, Sequence

import numpy as np

from . import _native, schedule
from .gate_list import GateList, defer_phases

DEFER_PHASES = os.environ.get("QB_DEFER_PHASES", "1") != "0"  # A/B switch of the R_Y * D rewrite (gate_list.defer_phases)


def rewritten(gates: GateList, drop_final_phases: bool = False) -> GateList:
    """The gate list the engine really plans.  When the caller only needs |psi_k|^2 of the result (``drop_final_phases``:
    diagonal observables, sampling -- BASELINE configs C1, C2, C4) the trailing phase of every uncontrolled gate is deferred
    into the next gate on its qubit (12 instead of 14 multiply-adds per amplitude pair) and whatever is still pending at the
    end of the circuit is dropped.  Callers that need the amplitudes themselves (Pauli sums with X / Y terms, statevector
    read-out, the segments of a sharded state) keep the circuit as written: re-applying the pending phases as one diagonal op
    per qubit costs more than the deferral saves (measured: 24-qubit TFIM 944 -> 686 evals/s)."""
    if not DEFER_PHASES or not drop_final_phases:
        return gates
    return GateList(gates.n_qubits, defer_phases(gates.ops, True), gates.n_params, gates.param_names)

_DTYPES = {"complex128": _native.QB_C128, "c128": _native.QB_C128, "complex64": _native.QB_C64, "c64": _native.QB_C64}


def _dtype_code(dtype) -> int:
    key = np.dtype(dtype).name if not isinstance(dtype, str) else dtype
    if key not in _DTYPES:
        raise ValueError(f"dtype must be complex128 or complex64, got {dtype!r}")
    return _DTYPES[key]


# Host-side planning is device independent: one encoded program per (circuit structure, tile / register bits, start kind) serves
# every engine of the process (multi-GPU primitives upload the same program to each device they use).
_encoded_plans: dict = {}
_encoded_lock = threading.Lock()


def encoded_plan(gates: GateList, tile_bits: int, reg_bits: int, from_zero_state: bool):
    """-> (n_sweeps, n_passes, n_pass_ops, (sweeps, passes, pass_ops, angles, init_ops)) of ``schedule.plan_circuit``."""
    key = (int(tile_bits), int(reg_bits), bool(from_zero_state), gates.structure_key())
    with _encoded_lock:
        hit = _encoded_plans.get(key)
    if hit is not None:
        return hit
    plan = schedule.plan_circuit(gates.ops, gates.n_qubits, tile_bits=tile_bits, reg_bits=reg_bits, product_prefix=from_zero_state)
    arrays = schedule.encode_plan(plan, gates.ops)
    hit = (len(arrays[0]), len(arrays[1]), sum(s.n_ops for s in plan.sweeps), arrays)
    with _encoded_lock:
        if len(_encoded_plans) > 4096:
            _encoded_plans.clear()
        _encoded_plans[key] = hit
    return hit


class PlanHandle:
    __slots__ = ("plan_id", "n_qubits", "n_params", "n_ops", "n_sweeps", "n_passes", "dtype", "prefix", "__weakref__")

    def __init__(self, plan_id, n_qubits, n_params, n_ops, n_sweeps, n_passes, dtype):
        self.plan_id, self.n_qubits, self.n_params = plan_id, n_qubits, n_params
        self.n_ops, self.n_sweeps, self.n_passes, self.dtype = n_ops, n_sweeps, n_passes, dtype
        self.prefix = None  # PlanHandle of the parameter-free prefix this plan starts from (kept alive with it)


class HamiltonianHandle:
    __slots__ = ("ham_id", "n_qubits", "diagonal", "z_masks", "coeffs", "n_terms", "__weakref__")

    def __init__(self, ham_id, n_qubits, diagonal, z_masks, coeffs, n_terms):
        self.ham_id, self.n_qubits, self.diagonal = ham_id, n_qubits, diagonal
        self.z_masks, self.coeffs, self.n_terms = z_masks, coeffs, n_terms


class ObservablesHandle:
    __slots__ = ("obs_id", "n_qubits", "n_obs", "diagonal", "n_terms", "__weakref__")

    def __init__(self, obs_id, n_qubits, n_obs, diagonal, n_terms):
        self.obs_id, self.n_qubits, self.n_obs, self.diagonal, self.n_terms = obs_id, n_qubits, n_obs, diagonal, n_terms


def operator_terms(operator):
    """``SparsePauliOp``-like -> (n_qubits, x_masks, z_masks, coeffs) via the Qiskit API ``to_list()``
    (labels little-endian, right-most char = qubit 0)."""
    if hasattr(operator, "masks") and hasattr(operator, "num_qubits"):
        x, z, c = operator.masks()
        return int(operator.num_qubits), x, z, c
    if not hasattr(operator, "to_list"):
        raise TypeError(f"cannot extract Pauli terms from {type(operator).__name__}; a SparsePauliOp is required")
    from .operators import SparsePauliOp

    items = operator.to_list()
    op = SparsePauliOp.from_list(items, num_qubits=int(operator.num_qubits))
    x, z, c = op.masks()
    return op.num_qubits, x, z, c


def merge_duplicate_terms(x, z, c):
    """Sum the coefficients of identical (x, z) Pauli strings, keeping first-appearance order (the reference's JSSP encoder emits
    346 raw terms for 84 distinct strings at 26 qubits: job_shop_scheduling/domain_wall_hamiltonian_encoder.py:189-230)."""
    x = np.asarray(x, dtype=np.uint64)
    z = np.asarray(z, dtype=np.uint64)
    c = np.asarray(c, dtype=complex)
    if x.size < 2:
        return x, z, c
    keys = np.stack([x, z], axis=1)
    uniq, first, inverse = np.unique(keys, axis=0, return_index=True, return_inverse=True)
    if len(uniq) == x.size:
        return x, z, c
    inverse = np.asarray(inverse).reshape(-1)
    summed = np.zeros(len(uniq), dtype=complex)
    np.add.at(summed, inverse, c)
    order = np.argsort(first)
    return uniq[order, 0].copy(), uniq[order, 1].copy(), summed[order]


def observable_union(x, z, c, offsets):
    """The combination ``qb_observables_create`` builds from observable j's terms ``offsets[j] .. offsets[j+1]-1``: the distinct
    (x, z) strings in first-appearance order and CSR rows over them -> (ux, uz, row_begin, cols, coeffs), each row in ascending
    string order with the real parts of duplicate strings summed (every string is Hermitian, so Re(c) is all that counts)."""
    index_of: dict = {}
    ux, uz, row_begin, cols, coeffs = [], [], [0], [], []
    for j in range(len(offsets) - 1):
        row: dict = {}
        for t in range(int(offsets[j]), int(offsets[j + 1])):
            key = (int(x[t]), int(z[t]))
            u = index_of.setdefault(key, len(ux))
            if u == len(ux):
                ux.append(key[0]), uz.append(key[1])
            row[u] = row.get(u, 0.0) + float(np.real(c[t]))
        for u in sorted(row):
            cols.append(u), coeffs.append(row[u])
        row_begin.append(len(cols))
    return (np.asarray(ux, dtype=np.uint64), np.asarray(uz, dtype=np.uint64), np.asarray(row_begin, dtype=np.int64),
            np.asarray(cols, dtype=np.int64), np.asarray(coeffs, dtype=np.float64))


def observable_terms(operators):
    """Operators of one width -> (n_qubits, x, z, coeffs, offsets): the concatenated terms, duplicates merged per operator."""
    operators = list(operators)
    if not operators:
        raise ValueError("an observable set needs at least one observable")
    xs, zs, cs, offsets, width = [], [], [], [0], None
    for op in operators:
        n, x, z, c = operator_terms(op)
        if width is not None and n != width:
            raise ValueError(f"observables of one set must act on the same number of qubits ({width} and {n})")
        width = n
        x, z, c = merge_duplicate_terms(x, z, c)
        xs.append(np.asarray(x, dtype=np.uint64)), zs.append(np.asarray(z, dtype=np.uint64)), cs.append(np.asarray(c, dtype=complex))
        offsets.append(offsets[-1] + len(c))
    return int(width), np.concatenate(xs), np.concatenate(zs), np.concatenate(cs), np.asarray(offsets, dtype=np.int64)


TOP_MAX_STATES = 1 << 20


def check_top_limits(max_states, min_probability) -> tuple[int, float]:
    """The limits of every top-states call: ``max_states`` in [1, 2^20], ``min_probability`` finite and >= 0 (ValueError otherwise)."""
    if isinstance(max_states, bool) or not isinstance(max_states, (int, np.integer)) or not 1 <= int(max_states) <= TOP_MAX_STATES:
        raise ValueError(f"max_states must be an integer in [1, 2^20], got {max_states!r}")
    p = float(min_probability)
    if not math.isfinite(p) or p < 0.0:
        raise ValueError(f"min_probability must be finite and >= 0, got {min_probability!r}")
    return int(max_states), p


MARGINAL_MAX_QUBITS = 26


def check_marginal_qubits(qubits, n_qubits: int) -> list:
    """The measured qubits of a marginal: distinct qubit indices of an ``n_qubits``-qubit state, 1 to 26 of them (the output holds
    2^m doubles per state: 512 MiB at the cap).  ValueError otherwise."""
    try:
        qs = [int(q) for q in qubits]
    except TypeError:
        raise ValueError(f"qubits must be a sequence of qubit indices, got {qubits!r}") from None
    if not 1 <= len(qs) <= MARGINAL_MAX_QUBITS:
        raise ValueError(f"a marginal measures 1 to {MARGINAL_MAX_QUBITS} qubits (2^m doubles per state), got {len(qs)}")
    if len(set(qs)) != len(qs) or not all(0 <= q < n_qubits for q in qs):
        raise ValueError(f"qubits must be distinct indices in [0, {n_qubits}), got {qs}")
    return qs


def top_select_new(n_qubits: int, max_states: int) -> _native.TopSelect:
    """A fresh top-states select of ``max_states`` entries over a state of ``n_qubits`` logical qubits (``qb_top_select_init``)."""
    sel = _native.TopSelect()
    _native.check(_native.load().qb_top_select_init(byref(sel), int(n_qubits), int(max_states)))
    return sel


def top_select_pick(sel: _native.TopSelect, counts) -> None:
    """Advance ``sel`` by the 256 bucket counts of its pass, summed over all shards (``qb_top_select_pick``, pure host code)."""
    c = np.ascontiguousarray(counts, dtype=np.uint64).reshape(-1)
    if c.size != 256:
        raise ValueError("a select pass has 256 bucket counts")
    _native.check(_native.load().qb_top_select_pick(byref(sel), _native.ptr(c)))


@functools.lru_cache(maxsize=256)
def pipeline_split_point(n: int, n_eff: int, tile_bits: int, sm_count: int) -> Optional[int]:
    """First-chunk size of the two-chunk pipelined submission of ``n`` evaluations of ``n_eff``-qubit states: the split (between
    a fifth and half of the list) that wastes the fewest partially filled waves of sweep CTAs -- a state contributes
    tiles / 4 CTAs (tiles / 8 from 2^13 tiles on), an SM holds 4 of them (2 with 2^12-amplitude tiles).  None: do not split
    (large states: the value conversion is noise next to the GPU time and the native call chunks by memory itself)."""
    if n < 8 or n_eff > 24:
        return None
    tiles = 1 << (n_eff - tile_bits)
    ctas = max(1, tiles >> min(3, n_eff - tile_bits))
    slots = sm_count * (4 if tile_bits <= 11 else 2)

    def waste(c: int) -> float:
        w = c * ctas / slots
        return (math.ceil(w) - w) if w >= 1 else 0.0

    return min(range(max(2, n // 5), n // 2 + 1), key=lambda c: (round(waste(c) + waste(n - c), 3), c))


class Engine:
    """One native context (one CUDA device, one stream).  Thread-safe."""

    def __init__(self, device: int = 0, dtype="complex128", stream: Optional[int] = None, workspace_limit: int = 0, reg_bits: Optional[int] = None, tile_bits: Optional[int] = None):
        self._lib = _native.load()
        self.device = int(device)
        self.dtype = "complex128" if _dtype_code(dtype) == _native.QB_C128 else "complex64"
        self._dtype_code = _dtype_code(dtype)
        self.reg_bits = int(reg_bits if reg_bits is not None else os.environ.get("QB_REG_BITS", schedule.REG_BITS))
        self.tile_bits = int(tile_bits if tile_bits is not None else os.environ.get("QB_TILE_BITS", schedule.TILE_BITS))
        handle = c_void_p()
        _native.check(self._lib.qb_context_create(self.device, c_void_p(stream) if stream else None, byref(handle)))
        self._ctx = handle
        self._eval_fn = ctypes.cast(self._lib.qb_evaluate_expectation, c_void_p)  # handed to the marshalling helper
        self._lock = threading.Lock()
        self._plan_cache: dict = {}
        self._prefix_bytes = 0
        self._prefix_budget = int(os.environ.get("QB_PREFIX_CACHE_MB", 16384)) << 20  # device memory for cached prefix states
        # two-chunk pipelined submission of large lists: hides the list -> float64 conversion of the second chunk behind the first
        # chunk's GPU work.  With the C marshalling helper the conversion is 10x cheaper and the extra submission costs more
        # than it hides (measured 26.3 k vs 27.8 k evals/s end to end), so it is only used on the NumPy conversion path.
        self._pipeline = os.environ.get("QB_PIPELINE", "0" if _native.pyhelper() else "1") != "0"
        self._submit_lock = threading.Lock()
        self._sm_count = max(1, int(self._lib.qb_context_sm_count(self._ctx)))
        self._finalizer = weakref.finalize(self, Engine._destroy, self._lib, handle)
        if workspace_limit:
            _native.check(self._lib.qb_context_set_workspace_limit(self._ctx, int(workspace_limit)))

    @staticmethod
    def _destroy(lib, handle):
        lib.qb_context_destroy(handle)

    def close(self):
        self._finalizer()

    # ------------------------------------------------------------------ introspection
    @property
    def stream(self) -> int:
        return int(self._lib.qb_context_stream(self._ctx) or 0)

    @property
    def launch_count(self) -> int:
        return int(self._lib.qb_context_launch_count(self._ctx))

    def synchronize(self):
        _native.check(self._lib.qb_context_synchronize(self._ctx))

    @property
    def workspace_bytes(self) -> int:
        """Statevector workspace of this device; a state larger than this has to be sharded over several GPUs."""
        return int(self._lib.qb_context_workspace(self._ctx))

    def set_index_width(self, bits: int):
        """64: run the 64-bit-index sweep kernels (what > 31 local qubits use) at any size; 32: automatic."""
        _native.check(self._lib.qb_context_set_index_width(self._ctx, int(bits)))

    # ------------------------------------------------------------------ compilation
    def compile_with_prefix_reuse(self, gates: GateList, dtype=None, min_prefix_ops: int = 4, drop_final_phases: bool = False) -> PlanHandle:
        """Like ``compile``, but a leading run of parameter-free ops (the numerically bound layers of a partially
        parameterised EVQE circuit: evqe/evolutionary_algorithm/individual.py:288-322) is compiled as a separate plan
        whose resulting state is computed once and cached on the device; every evaluation then only applies the
        remaining ops (SURVEY.md section 8f-1).  The returned handle owns the cached state: it is not shared through
        the structural plan cache and is released with the handle.  Falls back to ``compile`` when there is nothing
        to reuse or the cached states would exceed a quarter of the workspace budget."""
        gates = rewritten(gates, drop_final_phases)  # before the split: the pending phases cross the prefix / suffix boundary
        split = 0
        for op in gates.ops:
            if any(a.slot >= 0 or a.slot2 >= 0 for a in op.angles):
                break
            split += 1
        state_bytes = (16 if (self._dtype_code if dtype is None else _dtype_code(dtype)) == _native.QB_C128 else 8) << max(gates.n_qubits, self.tile_bits)
        if split < min_prefix_ops or split == len(gates.ops) or gates.n_params == 0:
            return self.compile(gates, dtype, defer=False)
        with self._lock:
            fits = self._prefix_bytes + state_bytes <= self._prefix_budget
            if fits:
                self._prefix_bytes += state_bytes
        if not fits:  # (compile takes the lock itself: not inside the block above)
            return self.compile(gates, dtype, defer=False)
        try:
            prefix = self.compile(GateList(gates.n_qubits, list(gates.ops[:split]), 0, ()), dtype, from_zero_state=True, defer=False)
            suffix = self.compile(GateList(gates.n_qubits, list(gates.ops[split:]), gates.n_params, gates.param_names), dtype, from_zero_state=False, cache=False, defer=False)
            _native.check(self._lib.qb_plan_set_prefix(self._ctx, suffix.plan_id, prefix.plan_id))
        except BaseException:
            self._release_prefix_bytes(state_bytes)  # nothing was cached: give the budget back
            raise
        suffix.prefix = prefix
        weakref.finalize(suffix, self._release_prefix_bytes, state_bytes)
        return suffix

    def _release_prefix_bytes(self, nbytes):
        with self._lock:
            self._prefix_bytes -= nbytes

    def compile(self, gates: GateList, dtype=None, from_zero_state: bool = True, cache: bool = True, defer: bool = True, drop_final_phases: bool = False) -> PlanHandle:
        """``from_zero_state=False``: the plan will be applied to an existing state (no product-state prefix).
        ``drop_final_phases=True``: the caller only needs |psi_k|^2 of the result (diagonal observable, sampling): the
        diagonal phases left pending at the end of the circuit are not applied (``rewritten``)."""
        code = self._dtype_code if dtype is None else _dtype_code(dtype)
        if defer:
            gates = rewritten(gates, drop_final_phases)
        key = (code, bool(from_zero_state), gates.structure_key())
        with self._lock:
            hit = self._plan_cache.get(key) if cache else None
        if hit is not None:
            return hit
        _, _, n_pass_ops, (sweeps, passes, pass_ops, angles, init_ops) = encoded_plan(gates, self.tile_bits, self.reg_bits, from_zero_state)
        plan_id = c_int64()
        _native.check(
            self._lib.qb_plan_create(
                self._ctx, gates.n_qubits, code, self.tile_bits, self.reg_bits, gates.n_params, len(gates.ops), _native.ptr(angles), len(sweeps), _native.ptr(sweeps),
                len(passes), _native.ptr(passes), n_pass_ops, _native.ptr(pass_ops), _native.ptr(init_ops), byref(plan_id),
            )
        )
        handle = PlanHandle(plan_id.value, gates.n_qubits, gates.n_params, len(gates.ops), len(sweeps), len(passes), code)
        weakref.finalize(handle, self._release_plan, self._lib, self._ctx, plan_id.value, self._finalizer)
        if cache:
            with self._lock:
                if len(self._plan_cache) > 4096:
                    self._plan_cache.clear()
                self._plan_cache[key] = handle
        return handle

    @staticmethod
    def _release_plan(lib, ctx, plan_id, engine_finalizer):
        if engine_finalizer.alive:
            lib.qb_plan_destroy(ctx, plan_id)

    def hamiltonian(self, operator, build_table: Optional[bool] = None) -> HamiltonianHandle:
        n, x, z, c = operator_terms(operator)
        x, z, c = merge_duplicate_terms(x, z, c)  # the reference's encoders emit each (x, z) string many times over
        x = np.ascontiguousarray(x, dtype=np.uint64)
        z = np.ascontiguousarray(z, dtype=np.uint64)
        cre = np.ascontiguousarray(c.real, dtype=np.float64)
        cim = np.ascontiguousarray(c.imag, dtype=np.float64)
        diagonal = not bool(np.any(x))
        n_diag = int(np.count_nonzero(x == 0))
        table_bytes = 8 << max(n, self.tile_bits)
        if build_table is None:
            # a table costs 8 B * 2^n once and turns the per-amplitude cost from O(terms) into one load; above a sixteenth of
            # the statevector workspace (30 qubits on a 180 GB B200) the terms are evaluated on the fly instead
            build_table = n_diag > 8 and table_bytes <= self.workspace_bytes // 16
        elif build_table and table_bytes > self.workspace_bytes // 2:
            raise ValueError(f"a diagonal table of {table_bytes >> 30} GiB does not fit next to the statevector workspace ({self.workspace_bytes >> 30} GiB)")
        ham_id = c_int64()
        _native.check(
            self._lib.qb_hamiltonian_create(self._ctx, n, len(cre), _native.ptr(x), _native.ptr(z), _native.ptr(cre), _native.ptr(cim), int(bool(build_table)), byref(ham_id))
        )
        handle = HamiltonianHandle(ham_id.value, n, diagonal, z[x == 0].copy(), cre[x == 0].copy(), len(cre))
        weakref.finalize(handle, self._release_ham, self._lib, self._ctx, ham_id.value, self._finalizer)
        return handle

    @staticmethod
    def _release_ham(lib, ctx, ham_id, engine_finalizer):
        if engine_finalizer.alive:
            lib.qb_hamiltonian_destroy(ctx, ham_id)

    def observables(self, operators: Sequence) -> ObservablesHandle:
        """Device form of several observables of one width, evaluated together by ``expectation_many``: the union of their
        distinct Pauli strings, grouped by x mask (``qb_observables_create``)."""
        width, x, z, c, offs = observable_terms(operators)
        x = np.ascontiguousarray(x, dtype=np.uint64)
        z = np.ascontiguousarray(z, dtype=np.uint64)
        cre = np.ascontiguousarray(c.real, dtype=np.float64)
        cim = np.ascontiguousarray(c.imag, dtype=np.float64)
        pad = lambda a: a if a.size else np.zeros(1, dtype=a.dtype)  # (valid pointers for a set of empty operators)
        obs_id = c_int64()
        _native.check(
            self._lib.qb_observables_create(self._ctx, width, len(offs) - 1, _native.ptr(offs), _native.ptr(pad(x)), _native.ptr(pad(z)),
                                            _native.ptr(pad(cre)), _native.ptr(pad(cim)), byref(obs_id))
        )
        n_terms = len(observable_union(x, z, c, offs)[0])
        handle = ObservablesHandle(obs_id.value, width, len(offs) - 1, not bool(np.any(x)), n_terms)
        weakref.finalize(handle, self._release_observables, self._lib, self._ctx, obs_id.value, self._finalizer)
        return handle

    @staticmethod
    def _release_observables(lib, ctx, obs_id, engine_finalizer):
        if engine_finalizer.alive:
            lib.qb_observables_destroy(ctx, obs_id)

    # ------------------------------------------------------------------ batched evaluation
    @staticmethod
    def _pack(plans: Sequence[PlanHandle], params: Sequence[Sequence[float]]):
        if len(plans) != len(params):
            raise ValueError(f"{len(plans)} circuits but {len(params)} parameter vectors")
        if len(plans) == 1:  # the optimizer loop's call: one circuit, one parameter vector
            row, want = params[0], plans[0].n_params
            helper = _native.pyhelper() if isinstance(row, (list, tuple)) and len(row) == want and want else None
            flat = None
            if helper:
                flat = np.empty(want, dtype=np.float64)
                if helper.qb_pack_rows((row,), flat.ctypes.data, np.array([want], dtype=np.int64).ctypes.data, 1) != want:
                    flat = None
            if flat is None:
                flat = np.asarray(row, dtype=np.float64).reshape(-1)
            if flat.size != want:
                raise ValueError(f"circuit 0 has {want} parameters but {flat.size} values were given")
            return np.array([plans[0].plan_id], dtype=np.int64), (flat if flat.size else np.zeros(1, dtype=np.float64)), np.array([0, flat.size], dtype=np.int64)
        ids = np.fromiter((p.plan_id for p in plans), dtype=np.int64, count=len(plans))
        offsets = np.zeros(len(plans) + 1, dtype=np.int64)
        if isinstance(params, np.ndarray) and params.ndim == 2 and params.dtype == np.float64:
            # one block of equally long parameter vectors (batched optimizer evaluation): no per-row conversion
            width = params.shape[1]
            for i, pl in enumerate(plans):
                if pl.n_params != width:
                    raise ValueError(f"circuit {i} has {pl.n_params} parameters but {width} values were given")
            offsets[1:] = np.arange(1, len(plans) + 1, dtype=np.int64) * width
            flat = np.ascontiguousarray(params).reshape(-1)
            return ids, (flat if flat.size else np.zeros(1, dtype=np.float64)), offsets
        helper = _native.pyhelper() if isinstance(params, (list, tuple)) and params and isinstance(params[0], (list, tuple)) else None
        if helper:
            # the reference's list[list[float]]: one C pass over the Python objects instead of one NumPy call per row
            expected = np.fromiter((p.n_params for p in plans), dtype=np.int64, count=len(plans))
            np.cumsum(expected, out=offsets[1:])
            flat = np.empty(max(1, int(offsets[-1])), dtype=np.float64)
            got = helper.qb_pack_rows(params, _native.ptr(flat), _native.ptr(expected), len(plans))
            if got == offsets[-1]:
                return ids, flat, offsets
            if -len(plans) <= got < 0:
                i = int(-got - 1)
                raise ValueError(f"circuit {i} has {plans[i].n_params} parameters but {len(params[i])} values were given")
            offsets[:] = 0  # rows the helper cannot read (nested arrays, exotic number types): the NumPy path below decides
        chunks = []
        for i, (pl, vals) in enumerate(zip(plans, params)):
            arr = np.asarray(vals, dtype=np.float64).reshape(-1)
            if arr.size != pl.n_params:
                raise ValueError(f"circuit {i} has {pl.n_params} parameters but {arr.size} values were given")
            chunks.append(arr)
            offsets[i + 1] = offsets[i] + arr.size
        flat = np.concatenate(chunks) if chunks and offsets[-1] else np.zeros(1, dtype=np.float64)
        return ids, np.ascontiguousarray(flat), offsets

    def expectation(self, plans: Sequence[PlanHandle], params: Sequence[Sequence[float]], ham: HamiltonianHandle) -> np.ndarray:
        if not plans:
            return np.zeros(0)
        if len(plans) != len(params):
            raise ValueError(f"{len(plans)} circuits but {len(params)} parameter vectors")
        if len(plans) == 1:  # the optimizer loop's call: one native-helper call packs the row and evaluates it
            row, plan = params[0], plans[0]
            helper = _native.pyhelper() if type(row) in (list, tuple) else None
            if helper:
                r = helper.qb_single_expectation(self._eval_fn, self._ctx, plan.plan_id, plan.n_params, row, ham.ham_id)
                if type(r) is float:
                    return np.array((r,))
                if r == -1000:
                    raise ValueError(f"circuit 0 has {plan.n_params} parameters but {len(row)} values were given")
                if r != -2000:  # (-2000: a row the helper cannot read -- the NumPy path below decides)
                    _native.check(r)
        out = np.empty(len(plans), dtype=np.float64)
        split = self._pipeline_split(plans, params)
        if split is None:
            ids, flat, offsets = self._pack(plans, params)
            _native.check(self._lib.qb_evaluate_expectation(self._ctx, len(plans), _native.ptr(ids), _native.ptr(flat), _native.ptr(offsets), ham.ham_id, _native.ptr(out)))
            return out
        # pipelined submission: the GPU starts on the first chunk while the parameter lists of the second are still being
        # converted to float64 arrays (for a population of Python float lists that conversion is most of the host time)
        with self._submit_lock:
            try:
                for lo, hi in ((0, split), (split, len(plans))):
                    ids, flat, offsets = self._pack(plans[lo:hi], params[lo:hi])
                    _native.check(self._lib.qb_evaluate_expectation_submit(self._ctx, hi - lo, _native.ptr(ids), _native.ptr(flat), _native.ptr(offsets), ham.ham_id))
            except _native.QbError as exc:
                self._lib.qb_evaluate_expectation_collect(self._ctx, 0, None)  # drain whatever was queued
                if exc.code != _native.QB_ERR_MEMORY:
                    raise
                split = None  # a chunk does not fit the statevector workspace: the one-shot call chunks by memory itself
            except Exception:
                self._lib.qb_evaluate_expectation_collect(self._ctx, 0, None)
                raise
            if split is not None:
                _native.check(self._lib.qb_evaluate_expectation_collect(self._ctx, len(plans), _native.ptr(out)))
                return out
        ids, flat, offsets = self._pack(plans, params)
        _native.check(self._lib.qb_evaluate_expectation(self._ctx, len(plans), _native.ptr(ids), _native.ptr(flat), _native.ptr(offsets), ham.ham_id, _native.ptr(out)))
        return out

    def expectation_submit(self, plans: Sequence[PlanHandle], params: Sequence[Sequence[float]], ham: HamiltonianHandle) -> int:
        """Queue the evaluation of a whole list on this engine's stream and return at once (``qb_evaluate_expectation_submit``);
        ``expectation_collect`` waits for it.  A caller that drives several devices submits to all of them first and collects
        afterwards, so the GPUs work concurrently without one Python thread per device.  The engine stays reserved for the
        caller between the two calls (other submitters wait).  Raises ``QbError`` (``QB_ERR_MEMORY``) when the list does not
        fit the statevector workspace in one piece -- use ``expectation`` then, which chunks by memory."""
        if len(plans) != len(params):
            raise ValueError(f"{len(plans)} circuits but {len(params)} parameter vectors")
        ids, flat, offsets = self._pack(plans, params)
        self._submit_lock.acquire()
        try:
            _native.check(self._lib.qb_evaluate_expectation_submit(self._ctx, len(plans), _native.ptr(ids), _native.ptr(flat), _native.ptr(offsets), ham.ham_id))
        except BaseException:
            self._lib.qb_evaluate_expectation_collect(self._ctx, 0, None)  # drain whatever was queued
            self._submit_lock.release()
            raise
        return len(plans)

    def expectation_collect(self, count: int) -> np.ndarray:
        """Wait for the list queued by ``expectation_submit`` and return its ``count`` values in submission order."""
        out = np.empty(count, dtype=np.float64)
        try:
            _native.check(self._lib.qb_evaluate_expectation_collect(self._ctx, count, _native.ptr(out)))
        finally:
            self._submit_lock.release()
        return out

    def _pipeline_split(self, plans: Sequence[PlanHandle], params) -> Optional[int]:
        """Size of the first chunk of a two-chunk pipelined submission, or None to submit in one piece.  Worth it when the
        parameter values arrive as Python sequences (not arrays) and the batch is large; the split point is chosen so that
        both chunks fill whole waves of sweep CTAs (tiles / 4 CTAs per state, 4 resident CTAs per SM)."""
        n = len(plans)
        if n < 8 or not self._pipeline or isinstance(params, np.ndarray) or isinstance(params[0], np.ndarray):
            return None
        if sum(p.n_params for p in plans) < 2048:
            return None
        return pipeline_split_point(n, max(plans[0].n_qubits, self.tile_bits), self.tile_bits, self._sm_count)

    def sample(self, plans: Sequence[PlanHandle], params: Sequence[Sequence[float]], shots: int, uniforms: np.ndarray) -> np.ndarray:
        if not plans:
            return np.zeros((0, shots), dtype=np.int64)
        ids, flat, offsets = self._pack(plans, params)
        uniforms = np.ascontiguousarray(uniforms, dtype=np.float64).reshape(len(plans), shots)
        out = np.empty((len(plans), shots), dtype=np.int64)
        _native.check(self._lib.qb_sample(self._ctx, len(plans), _native.ptr(ids), _native.ptr(flat), _native.ptr(offsets), int(shots), _native.ptr(uniforms), _native.ptr(out)))
        return out

    def cvar(self, plans: Sequence[PlanHandle], params: Sequence[Sequence[float]], ham: HamiltonianHandle, alpha: float) -> np.ndarray:
        """Exact CVaR(alpha) of the diagonal ``ham`` on every circuit's full distribution |psi|^2, no shots
        (``qb_evaluate_cvar``: ``expectation.lower_tail_expectation_arrays`` over all 2^n basis states)."""
        if not plans:
            return np.zeros(0)
        ids, flat, offsets = self._pack(plans, params)  # (raises ValueError for a length mismatch, as in expectation / sample)
        out = np.empty(len(plans), dtype=np.float64)
        _native.check(self._lib.qb_evaluate_cvar(self._ctx, len(plans), _native.ptr(ids), _native.ptr(flat), _native.ptr(offsets), ham.ham_id, float(alpha), _native.ptr(out)))
        return out

    def top_states(self, plans: Sequence[PlanHandle], params: Sequence[Sequence[float]], max_states: int, min_probability: float = 0.0) -> list:
        """The most probable basis states of every circuit's state, exactly, without shots or a copy of the state
        (``qb_top_states``): per circuit (int64 logical indices, float64 probabilities), descending probability, ties in ascending
        index, at most ``max_states`` entries with p > 0 and p >= ``min_probability``."""
        max_states, min_probability = check_top_limits(max_states, min_probability)
        if not plans:
            return []
        ids, flat, offsets = self._pack(plans, params)
        counts = np.empty(len(plans), dtype=np.int64)
        idx = np.empty((len(plans), max_states), dtype=np.int64)
        probs = np.empty((len(plans), max_states), dtype=np.float64)
        _native.check(self._lib.qb_top_states(self._ctx, len(plans), _native.ptr(ids), _native.ptr(flat), _native.ptr(offsets), max_states, min_probability,
                                              _native.ptr(counts), _native.ptr(idx), _native.ptr(probs)))
        return [(idx[i, : counts[i]].copy(), probs[i, : counts[i]].copy()) for i in range(len(plans))]

    def marginal_probabilities(self, plans: Sequence[PlanHandle], params: Sequence[Sequence[float]], qubits: Sequence[int]) -> np.ndarray:
        """Exact marginal probabilities of every circuit's state on ``qubits``, without shots or a copy of the state
        (``qb_marginal_probabilities``): float64 [len(plans), 2^m], bit j of the column index = qubit ``qubits[j]`` (the convention of
        ``Statevector.probabilities(qargs)``).  Deterministic: the same state gives the same bits."""
        if not plans:
            return np.zeros((0, 1 << len(qubits)))
        qs = np.asarray(check_marginal_qubits(qubits, plans[0].n_qubits), dtype=np.int32)
        ids, flat, offsets = self._pack(plans, params)
        out = np.empty((len(plans), 1 << qs.size), dtype=np.float64)
        _native.check(self._lib.qb_marginal_probabilities(self._ctx, len(plans), _native.ptr(ids), _native.ptr(flat), _native.ptr(offsets), int(qs.size),
                                                          _native.ptr(qs), _native.ptr(out)))
        return out

    def expectation_many(self, plans: Sequence[PlanHandle], params: Sequence[Sequence[float]], handle: ObservablesHandle) -> np.ndarray:
        """Re <psi_i|H_j|psi_i> of every circuit and every observable of ``handle``: float64 array [len(plans), n_obs], each
        distinct Pauli string reduced once per state (``qb_evaluate_observables``)."""
        if not plans:
            return np.zeros((0, handle.n_obs))
        ids, flat, offsets = self._pack(plans, params)
        out = np.empty((len(plans), handle.n_obs), dtype=np.float64)
        _native.check(self._lib.qb_evaluate_observables(self._ctx, len(plans), _native.ptr(ids), _native.ptr(flat), _native.ptr(offsets), handle.obs_id, _native.ptr(out)))
        return out

    def statevector(self, plan: PlanHandle, params: Sequence[float]) -> np.ndarray:
        vals = np.ascontiguousarray(np.asarray(params, dtype=np.float64).reshape(-1))
        if vals.size != plan.n_params:
            raise ValueError(f"circuit has {plan.n_params} parameters but {vals.size} values were given")
        out = np.empty(1 << plan.n_qubits, dtype=np.complex128)
        buf = vals if vals.size else np.zeros(1)
        _native.check(self._lib.qb_statevector(self._ctx, plan.plan_id, _native.ptr(buf), int(vals.size), _native.ptr(out)))
        return out

    def diag_energies(self, ham: HamiltonianHandle, states: np.ndarray) -> np.ndarray:
        states = np.ascontiguousarray(states, dtype=np.uint64).reshape(-1)
        out = np.empty(states.size, dtype=np.float64)
        if states.size:
            _native.check(self._lib.qb_hamiltonian_diag_energies(self._ctx, ham.ham_id, states.size, _native.ptr(states), _native.ptr(out)))
        return out

    def resident_batch(self, plans: Sequence[PlanHandle], ham: Optional[HamiltonianHandle]) -> "ResidentBatch":
        return ResidentBatch(self, plans, ham)

    # ------------------------------------------------------------------ device-pointer entry points
    def apply_plan_device(self, plan: PlanHandle, params: Sequence[float], state_ptr: int, init_zero_state: bool, index_offset: int = 0):
        vals = np.ascontiguousarray(np.asarray(params, dtype=np.float64).reshape(-1))
        buf = vals if vals.size else np.zeros(1)
        _native.check(self._lib.qb_apply_plan_device(self._ctx, plan.plan_id, _native.ptr(buf), int(vals.size), c_void_p(state_ptr), int(init_zero_state), int(index_offset)))

    def expectation_device(self, ham: HamiltonianHandle, dtype, n_local: int, state_ptr: int, index_offset: int = 0) -> float:
        out = c_double()
        _native.check(self._lib.qb_expectation_device(self._ctx, ham.ham_id, _dtype_code(dtype), int(n_local), c_void_p(state_ptr), int(index_offset), byref(out)))
        return out.value

    def cvar_select_device(self, ham: HamiltonianHandle, dtype, n_local: int, state_ptr: int, index_offset: int, cache_ptr: int, cache_mode: int,
                           e_prefix: int, e_free: int, digit_kind: int, positions: Sequence[int], idx_mask: int, idx_value: int):
        """One select pass of the sharded exact CVaR on a caller-owned shard (``qb_cvar_select_device``, include/queasars_b200.h) ->
        (sums float64 [2, 256]: mass, sum p * E;  ints uint64 [4, 256]: count, min / max energy key, least physical index)."""
        pos = np.zeros(8, dtype=np.int32)
        pos[: len(positions)] = list(positions)
        bits = len(positions) if digit_kind == 1 else 8
        sums = np.empty((2, 256), dtype=np.float64)
        ints = np.empty((4, 256), dtype=np.uint64)
        _native.check(self._lib.qb_cvar_select_device(self._ctx, ham.ham_id, _dtype_code(dtype), int(n_local), c_void_p(state_ptr), int(index_offset),
                                                      c_void_p(cache_ptr or None), int(cache_mode), int(e_prefix), int(e_free), int(digit_kind), int(bits),
                                                      _native.ptr(pos), int(idx_mask), int(idx_value), _native.ptr(sums), _native.ptr(ints)))
        return sums, ints

    def top_select_device(self, dtype, n_local: int, state_ptr: int, index_offset: int, min_probability: float, sel: _native.TopSelect,
                          positions: Optional[Sequence[int]] = None) -> np.ndarray:
        """Bucket counts (uint64 [256]) of the select pass ``sel`` describes on a caller-owned shard (``qb_top_select_device``);
        ``positions[q]`` = physical bit position of logical qubit q (None: the identity)."""
        pos = None if positions is None else np.ascontiguousarray(positions, dtype=np.int32)
        out = np.empty(256, dtype=np.uint64)
        _native.check(self._lib.qb_top_select_device(self._ctx, _dtype_code(dtype), int(n_local), c_void_p(state_ptr), int(index_offset), float(min_probability),
                                                     byref(sel), None if pos is None else _native.ptr(pos), _native.ptr(out)))
        return out

    def top_collect_device(self, dtype, n_local: int, state_ptr: int, index_offset: int, min_probability: float, sel: _native.TopSelect,
                           positions: Optional[Sequence[int]], capacity: int):
        """This shard's entries up to the stop key of the finished select ``sel`` (``qb_top_collect_device``), in physical index
        order -> (int64 physical indices, float64 probabilities)."""
        pos = None if positions is None else np.ascontiguousarray(positions, dtype=np.int32)
        cap = max(1, int(capacity))
        idx = np.empty(cap, dtype=np.int64)
        probs = np.empty(cap, dtype=np.float64)
        count = c_int64()
        _native.check(self._lib.qb_top_collect_device(self._ctx, _dtype_code(dtype), int(n_local), c_void_p(state_ptr), int(index_offset), float(min_probability),
                                                      byref(sel), None if pos is None else _native.ptr(pos), int(capacity), byref(count), _native.ptr(idx),
                                                      _native.ptr(probs)))
        return idx[: count.value].copy(), probs[: count.value].copy()

    def marginal_device(self, dtype, n_local: int, state_ptr: int, index_offset: int, positions: Sequence[int]) -> np.ndarray:
        """This shard's part of a marginal (``qb_marginal_device``): float64 [2^m], bit j of the index = physical bit ``positions[j]``;
        rank bits (positions >= n_local) read their value from ``index_offset``."""
        pos = np.ascontiguousarray(positions, dtype=np.int32)
        out = np.empty(1 << pos.size, dtype=np.float64)
        _native.check(self._lib.qb_marginal_device(self._ctx, _dtype_code(dtype), int(n_local), c_void_p(state_ptr), int(index_offset), int(pos.size),
                                                   _native.ptr(pos), _native.ptr(out)))
        return out

    def swap_global_p2p(self, dtype, n_local: int, state_ptr: int, peer_ptrs: Sequence[int], rank: int, local_positions: Sequence[int]):
        """Launch the fused swap + all-to-all kernel (asynchronous on the engine's stream; see include/queasars_b200.h)."""
        world = len(peer_ptrs)
        ptrs = np.asarray([int(p) for p in peer_ptrs], dtype=np.uint64)
        lp = np.asarray(list(local_positions), dtype=np.int32)
        _native.check(self._lib.qb_swap_global_p2p(self._ctx, _dtype_code(dtype), int(n_local), c_void_p(state_ptr), _native.ptr(ptrs), world, int(rank), len(lp), _native.ptr(lp)))

    def swap_global_inplace_p2p(self, dtype, n_local: int, shard_ptrs: Sequence[int], rank: int, local_positions: Sequence[int]):
        """Launch the in-place exchange kernel on every rank's state buffer ``shard_ptrs`` (one buffer per rank; asynchronous on the
        engine's stream; the caller owns the before / after barriers of include/queasars_b200.h)."""
        world = len(shard_ptrs)
        ptrs = np.asarray([int(p) for p in shard_ptrs], dtype=np.uint64)
        lp = np.asarray(list(local_positions), dtype=np.int32)
        _native.check(self._lib.qb_swap_global_inplace_p2p(self._ctx, _dtype_code(dtype), int(n_local), _native.ptr(ptrs), world, int(rank), len(lp),
                                                           _native.ptr(lp)))

    # ------------------------------------------------------------------ device memory / peer mapping (sharded states)
    def device_alloc(self, nbytes: int) -> int:
        out = c_void_p()
        _native.check(self._lib.qb_device_alloc(self._ctx, int(nbytes), byref(out)))
        return int(out.value)

    def device_free(self, ptr: int):
        if self._finalizer.alive:
            _native.check(self._lib.qb_device_free(self._ctx, c_void_p(ptr)))

    def device_read(self, ptr: int, offset: int, out: np.ndarray):
        _native.check(self._lib.qb_device_read(self._ctx, c_void_p(ptr), int(offset), int(out.nbytes), _native.ptr(out)))
        return out

    def enable_peer_access(self, peer_device: int):
        _native.check(self._lib.qb_enable_peer_access(self._ctx, int(peer_device)))

    def ipc_export(self, ptr: int) -> bytes:
        buf = (ctypes.c_ubyte * 64)()
        _native.check(self._lib.qb_ipc_export(self._ctx, c_void_p(ptr), buf))
        return bytes(buf)

    def ipc_open(self, handle: bytes) -> int:
        buf = (ctypes.c_ubyte * 64).from_buffer_copy(handle)
        out = c_void_p()
        _native.check(self._lib.qb_ipc_open(self._ctx, buf, byref(out)))
        return int(out.value)

    def ipc_close(self, ptr: int):
        if self._finalizer.alive:
            _native.check(self._lib.qb_ipc_close(self._ctx, c_void_p(ptr)))

    def sample_device(self, dtype, n_local: int, state_ptr: int, uniforms: np.ndarray) -> np.ndarray:
        """searchsorted(cumsum(|psi|^2) / sum, uniforms, side='right') on a caller-owned device state (a shard)."""
        uniforms = np.ascontiguousarray(uniforms, dtype=np.float64).reshape(-1)
        out = np.empty(uniforms.size, dtype=np.int64)
        if uniforms.size:
            _native.check(self._lib.qb_sample_device(self._ctx, _dtype_code(dtype), int(n_local), c_void_p(state_ptr), int(uniforms.size), _native.ptr(uniforms), _native.ptr(out)))
        return out


class ResidentBatch:
    """A fixed list of circuits whose device buffers stay allocated: ``set_params`` (H2D), ``run`` (kernels
    only, asynchronous), ``read`` (D2H + sync).  Used by bench.py and by optimizer inner loops."""

    def __init__(self, engine: Engine, plans: Sequence[PlanHandle], ham: Optional[HamiltonianHandle]):
        self._engine = engine
        self._plans = list(plans)
        self._ham = ham
        ids = np.fromiter((p.plan_id for p in self._plans), dtype=np.int64, count=len(self._plans))
        batch_id = c_int64()
        _native.check(engine._lib.qb_batch_create(engine._ctx, len(self._plans), _native.ptr(ids), ham.ham_id if ham else 0, byref(batch_id)))
        self.batch_id = batch_id.value
        self._finalizer = weakref.finalize(self, ResidentBatch._destroy, engine._lib, engine._ctx, self.batch_id, engine._finalizer)

    @staticmethod
    def _destroy(lib, ctx, batch_id, engine_finalizer):
        if engine_finalizer.alive:
            lib.qb_batch_destroy(ctx, batch_id)

    def __len__(self):
        return len(self._plans)

    def set_params(self, params: Sequence[Sequence[float]]):
        _, flat, offsets = Engine._pack(self._plans, params)
        _native.check(self._engine._lib.qb_batch_set_params(self._engine._ctx, self.batch_id, _native.ptr(flat), _native.ptr(offsets)))
        return int(flat.nbytes if offsets[-1] else 0)

    def set_params_flat(self, flat: np.ndarray, offsets: np.ndarray):
        _native.check(self._engine._lib.qb_batch_set_params(self._engine._ctx, self.batch_id, _native.ptr(flat), _native.ptr(offsets)))

    def run(self):
        _native.check(self._engine._lib.qb_batch_run(self._engine._ctx, self.batch_id))

    def run_timed(self):
        """-> (ms per sweep launch, statevectors swept per launch); CUDA events on the engine's stream."""
        cap = 4096
        ms = np.zeros(cap, dtype=np.float32)
        states = np.zeros(cap, dtype=np.int32)
        n = ctypes.c_int()
        _native.check(self._engine._lib.qb_batch_run_timed(self._engine._ctx, self.batch_id, cap, _native.ptr(ms), _native.ptr(states), byref(n)))
        return ms[: n.value].astype(np.float64), states[: n.value].astype(np.int64)

    def read(self) -> np.ndarray:
        out = np.empty(len(self._plans), dtype=np.float64)
        _native.check(self._engine._lib.qb_batch_read(self._engine._ctx, self.batch_id, _native.ptr(out)))
        return out

    def stats(self) -> dict:
        a, b, c, d = c_int64(), c_int64(), c_int64(), c_int64()
        _native.check(self._engine._lib.qb_batch_stats(self._engine._ctx, self.batch_id, byref(a), byref(b), byref(c), byref(d)))
        return {"sweep_launches": a.value, "state_sweeps": b.value, "sweep_bytes": c.value, "kernel_launches": d.value}

    def close(self):
        self._finalizer()
