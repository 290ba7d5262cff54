"""One statevector sharded over several GPUs by its top ("global") qubits -- BASELINE config C5
(35 qubits complex128 = 512 GiB over 8 x B200).  New capability: the reference has no single-state scaling
mechanism (SURVEY.md section 5); the same `evaluate` semantics as the single-GPU engine are kept.

Layout: world = 2^g shards, shard r holds the 2^(n-g) amplitudes whose top g index bits equal r.  A *physical*
bit position p < n-g is local, p >= n-g is a rank bit.  Logical qubits are tracked through a permutation
(`position[q]`), so a swap is pure relabelling plus data movement:

  * gates whose target sits on a local position run the normal sweep kernel on the shard
    (``qb_apply_plan_device`` with ``index_offset = rank << n_local``: a control or diagonal target on a rank bit is
    a per-shard predicate, no communication);
  * before a gate that *targets* a rank bit, all g rank bits are exchanged with g local positions whose qubits are
    needed latest.  On GPUs the exchange is ONE kernel per shard (``qb_swap_global_p2p``): it streams the shard once and
    stores every amplitude straight into the GPU that owns it afterwards, at its final index, through peer-mapped
    buffers over NVLink 5 / NVSwitch -- the all-to-all is fused into the permutation, there is no pack pass, no staging
    copy and no unpack pass.  Two buffers of shard size are used in ping-pong.

Two drivers share the schedule (``_ShardedLogic``):

  ``ShardedStatevector``       one process per GPU (``torchrun``): collectives over ``torch.distributed``; the shard buffers are
                               cudaMalloc allocations made through the C-ABI and mapped into the peers with CUDA IPC handles
                               (``qb_ipc_export`` / ``qb_ipc_open``) exchanged by an all-gather.  ``QB_SWAP=nccl``, CPU / gloo
                               tests and systems without peer mapping use pack -> ``all_to_all_single`` -> unpack instead; the
                               reason is kept in ``swap_fallback_reason`` and reported by ``describe()``.
  ``LocalShardedStatevector``  ONE process driving all shards (the configuration behind ``evaluate_circuits``: the evaluators
                               route circuits too wide for one GPU here): one engine + worker thread per device,
                               ``cudaDeviceEnablePeerAccess`` instead of IPC, reductions on the host.

The shard-local arithmetic is delegated to a *backend* object (``apply``, ``diagonal_expectation``, ``pauli_expectation``,
``sample``, ``cvar_select``, ``swap_p2p``); the product default drives the CUDA engine.  Tests inject a NumPy backend to exercise the
multi-rank host logic on CPU with the gloo backend.
"""
from __future__ import annotations

import math
import os
from typing import Optional, Sequence

import numpy as np

from .gate_list import DENSE, GateList, KernelOp


def _remap(op: KernelOp, position: Sequence[int]) -> KernelOp:
    return KernelOp(op.kind, position[op.target], -1 if op.control < 0 else position[op.control], op.gamma, op.theta, op.phi, op.lam)


def _state_ptr(state) -> int:
    return state.data_ptr() if hasattr(state, "data_ptr") else int(state)


_SIGN = np.uint64(1 << 63)


def energy_keys(energies) -> np.ndarray:
    """Order-preserving uint64 image of float64 energies (``energy_key`` of qb_kernels.cuh): ascending keys are ascending
    energies, and -0.0 gets the key of +0.0 (a radix sort and ``numpy.argsort(kind="stable")`` treat them as tied)."""
    u = np.ascontiguousarray(energies, dtype=np.float64).view(np.uint64).copy()
    u[u == _SIGN] = 0
    return np.where((u >> np.uint64(63)) == 1, ~u, u | _SIGN)


def energy_from_key(key: int) -> float:
    """Inverse of ``energy_keys`` (a key of +-0.0 gives +0.0)."""
    key = int(key)
    u = key & ((1 << 63) - 1) if key >> 63 else ~key & ((1 << 64) - 1)
    return float(np.asarray([u], dtype=np.uint64).view(np.float64)[0])


class CudaShardBackend:
    """Runs the shard-local work on the CUDA engine.  ``state`` is a torch tensor (only its ``data_ptr`` and stream are used)
    or a raw device address."""

    def __init__(self, engine):
        self.engine = engine
        self._select_ham = None

    @staticmethod
    def _join_torch_stream(state):
        # the engine launches on its own stream: everything torch queued on this buffer (pack / unpack copies,
        # the NCCL all-to-all) has to be complete before the kernels touch it.  The native calls synchronise
        # their stream before returning, which orders the other direction.
        if hasattr(state, "device"):
            import torch

            torch.cuda.current_stream(state.device).synchronize()

    def apply(self, state, ops: list[KernelOp], params: np.ndarray, n_local: int, n_params: int, index_offset: int, init_zero: bool):
        # controls may sit on rank bits (>= n_local), so the single-register product-state prefix does not apply
        plan = self.engine.compile(GateList(n_local, ops, n_params, ()), from_zero_state=False)
        self._join_torch_stream(state)
        self.engine.apply_plan_device(plan, params, _state_ptr(state), init_zero, index_offset)

    def diagonal_expectation(self, state, z_masks: np.ndarray, coeffs: np.ndarray, n_total: int, n_local: int, index_offset: int) -> float:
        from .operators import SparsePauliOp

        op = SparsePauliOp._raw(n_total, [0] * len(z_masks), [int(z) for z in z_masks], [float(c) for c in coeffs])
        ham = self.engine.hamiltonian(op, build_table=False)
        self._join_torch_stream(state)
        return self.engine.expectation_device(ham, "complex128", n_local, _state_ptr(state), index_offset)

    def pauli_expectation(self, state, x_masks, z_masks, coeffs, n_total: int, n_local: int, index_offset: int) -> float:
        """Shard-local part of Re <psi| sum_t c_t P_t |psi> for terms whose X part only flips local qubits (z may reach
        rank bits: they enter through index_offset)."""
        from .operators import SparsePauliOp

        op = SparsePauliOp._raw(n_total, [int(x) for x in x_masks], [int(z) for z in z_masks], [complex(c) for c in coeffs])
        ham = self.engine.hamiltonian(op, build_table=False)
        self._join_torch_stream(state)
        return self.engine.expectation_device(ham, "complex128", n_local, _state_ptr(state), index_offset)

    def sample(self, state, uniforms: np.ndarray, n_local: int) -> np.ndarray:
        self._join_torch_stream(state)
        return self.engine.sample_device("complex128", n_local, _state_ptr(state), uniforms)

    def cvar_select(self, state, cache, cache_mode: int, z_masks, coeffs, n_total: int, n_local: int, index_offset: int, spec):
        """One select pass of ``_ShardedLogic.cvar`` on this shard (``qb_cvar_select_device``); ``cache`` is the idle spare buffer."""
        key = (n_total, tuple(int(z) for z in z_masks), tuple(float(c) for c in coeffs))
        if self._select_ham is None or self._select_ham[0] != key:  # one Hamiltonian for all passes of a call
            from .operators import SparsePauliOp

            op = SparsePauliOp._raw(n_total, [0] * len(key[1]), list(key[1]), list(key[2]))
            self._select_ham = (key, self.engine.hamiltonian(op, build_table=False))
        self._join_torch_stream(state)
        return self.engine.cvar_select_device(self._select_ham[1], "complex128", n_local, _state_ptr(state), index_offset,
                                              0 if cache is None else _state_ptr(cache), cache_mode, *spec)

    def swap_p2p(self, state, peer_ptrs: Sequence[int], n_local: int, rank: int, local_positions: Sequence[int]) -> None:
        """Fused swap + all-to-all into the peers' buffers; returns when this rank's stores have been issued and completed."""
        self._join_torch_stream(state)
        self.engine.swap_global_p2p("complex128", n_local, _state_ptr(state), peer_ptrs, rank, local_positions)
        self.engine.synchronize()


class _ShardedLogic:
    """Placement-independent part: qubit permutation, segmenting of a gate list into shard-local runs separated by global
    swaps, observables expressed through per-shard partial results.  Subclasses provide
      _apply(segment, params, n_params, fresh)   run shard-local ops on every shard this object drives
      _swap(lp)                                   exchange the g rank bits with local positions lp (data movement only)
      _sum_over_shards(fn)                        sum over all shards of fn(rank, state) -> float  (every caller gets the total)
      _shard_masses()                             |shard|^2 of all shards, ndarray [world]
      _select_pass(z, c, cache_mode, spec)        every shard's bucket arrays of one cvar select pass, in rank order
      _sample_shards(owner, local_u)              physical indices of the shots (owner[s] = shard of shot s), int64 [shots]"""

    def _init_logic(self, n_qubits: int, world: int, min_local: int):
        g = int(round(math.log2(world)))
        if 1 << g != world:
            raise ValueError("the number of shards must be a power of two")
        self.world = world
        self.n_qubits, self.n_global, self.n_local = n_qubits, g, n_qubits - g
        if self.n_local < max(min_local, 2 * g):
            raise ValueError(f"{n_qubits} qubits over {world} shards leaves only {self.n_local} local qubits")
        self.position = list(range(n_qubits))  # logical qubit -> physical bit position
        self.swaps_done = 0
        self.bytes_sent = 0
        self._fresh = True
        self.swap_fallback_reason: Optional[str] = None

    def reset(self) -> None:
        """Forget the current state: the next ``run`` starts from |0...0> with the identity qubit placement."""
        self.position = list(range(self.n_qubits))
        self._fresh = True

    # ------------------------------------------------------------------ global <-> local swap
    def _swap_all_global(self, local_positions: Sequence[int]) -> None:
        """Exchange the g rank bits with the local bit positions ``local_positions`` (ascending list of length g).
        Afterwards rank bit j holds what was at local_positions[j] and vice versa."""
        g, nl = self.n_global, self.n_local
        if g == 0:
            return
        lp = list(local_positions)
        assert len(lp) == g and len(set(lp)) == g and all(0 <= p < nl for p in lp) and lp == sorted(lp)
        self._swap(lp)
        for q in range(self.n_qubits):
            p = self.position[q]
            if p >= nl:
                self.position[q] = lp[p - nl]
            elif p in lp:
                self.position[q] = nl + lp.index(p)
        self.swaps_done += 1
        self.bytes_sent += (self.world - 1) * ((1 << nl) // self.world) * 16

    # ------------------------------------------------------------------ circuit execution
    def run(self, gates: GateList, params: Sequence[float]) -> None:
        """Apply the circuit to |0...0> (first call) or to the current state."""
        if gates.n_qubits != self.n_qubits:
            raise ValueError("circuit and sharded state act on different numbers of qubits")
        params = np.ascontiguousarray(np.asarray(params, dtype=np.float64).reshape(-1))
        remaining = list(gates.ops)
        nl = self.n_local
        while remaining or self._fresh:
            # Everything that can run with the current placement: ops whose dense target is local and that do not
            # depend on a deferred op (same reordering rule as the sweep planner: two ops commute when they act
            # diagonally on every qubit they share).  Ops targeting a rank bit are deferred and served by ONE swap.
            pend_dense: set[int] = set()
            pend_any: set[int] = set()
            segment, deferred = [], []
            for op in remaining:
                t, c = op.target, op.control
                dense = op.kind == DENSE
                blocked = (t in pend_any) if dense else (t in pend_dense)
                if c >= 0 and c in pend_dense:
                    blocked = True
                if not blocked and not (dense and self.position[t] >= nl):
                    segment.append(_remap(op, self.position))
                    continue
                deferred.append(op)
                if dense:
                    pend_dense.add(t)
                pend_any.add(t)
                if c >= 0:
                    pend_any.add(c)
            if segment or self._fresh:
                self._apply(segment, params, gates.n_params, self._fresh)
                self._fresh = False
            remaining = deferred
            if remaining:
                self._swap_all_global(self._choose_local_positions(remaining))

    def _choose_local_positions(self, upcoming: Sequence[KernelOp]) -> list[int]:
        """Local positions to give up: those whose qubits are targeted latest (or never) by the upcoming ops."""
        nl = self.n_local
        first_use = {}
        for t, op in enumerate(upcoming):
            if op.kind == DENSE and op.target not in first_use:
                first_use[op.target] = t
        if all(self.position[q] < nl for q in first_use):  # nothing upcoming targets a rank bit
            return list(range(nl - self.n_global, nl))
        logical_at = {self.position[q]: q for q in range(self.n_qubits)}
        candidates = sorted(range(nl), key=lambda p: (-first_use.get(logical_at[p], 1 << 30), -p))
        return sorted(candidates[: self.n_global])

    # ------------------------------------------------------------------ observables
    def _physical_mask(self, mask: int) -> int:
        m = 0
        for q in range(self.n_qubits):
            if (int(mask) >> q) & 1:
                m |= 1 << self.position[q]
        return m

    def diagonal_expectation(self, z_masks: Sequence[int], coeffs: Sequence[float]) -> float:
        """<psi| sum_t c_t Z^{z_t} |psi> ; every caller gets the global value (one reduction of a double)."""
        phys = np.asarray([self._physical_mask(z) for z in z_masks], dtype=np.uint64)
        cf = np.asarray(coeffs, dtype=np.float64)
        return float(self._sum_over_shards(lambda backend, state, offset: backend.diagonal_expectation(state, phys, cf, self.n_qubits, self.n_local, offset)))

    def norm_squared(self) -> float:
        return self.diagonal_expectation([0], [1.0])

    def expectation(self, operator) -> float:
        """Re <psi|H|psi> for a general Pauli sum (SparsePauliOp-like: ``masks()`` -> x, z, coeffs as in operators.py).
        Terms whose X part flips only local qubits are evaluated shard-locally (Z factors on rank bits are per-shard
        signs); for the others ONE global swap brings the flipped rank bits down first, giving up local positions that
        no remaining term flips.  Every caller gets the global value."""
        from .engine import operator_terms

        n, xs, zs, cs = operator_terms(operator)
        if n != self.n_qubits:
            raise ValueError("operator and sharded state act on different numbers of qubits")
        todo = [(int(x), int(z), complex(c)) for x, z, c in zip(xs, zs, cs)]
        total = 0.0
        rank_bits = ((1 << self.n_global) - 1) << self.n_local
        for attempt in range(3):
            now = [t for t in todo if not (self._physical_mask(t[0]) & rank_bits)]
            todo = [t for t in todo if self._physical_mask(t[0]) & rank_bits]
            if now:
                px, pz, pc = [self._physical_mask(t[0]) for t in now], [self._physical_mask(t[1]) for t in now], [t[2] for t in now]
                total += self._sum_over_shards(lambda backend, state, offset: backend.pauli_expectation(state, px, pz, pc, self.n_qubits, self.n_local, offset))
            if not todo:
                break
            flipped = 0
            for x, _, _ in todo:
                flipped |= self._physical_mask(x)
            free = [p for p in range(self.n_local - 1, -1, -1) if not (flipped >> p) & 1]
            if attempt == 2 or len(free) < self.n_global:
                raise NotImplementedError("a Pauli term flips more qubits than fit one shard next to the rank bits")
            self._swap_all_global(sorted(free[: self.n_global]))
        return float(total)

    def cvar(self, z_masks: Sequence[int], coeffs: Sequence[float], alpha: float, cache: bool = True) -> tuple[float, int]:
        """Exact CVaR(alpha) of the diagonal Hamiltonian sum_t c_t Z^{z_t} on the whole distribution |psi|^2, no shots:
        ``expectation.lower_tail_expectation_arrays`` (the single-GPU ``Engine.cvar``) without gathering or sorting anything.
        Returns (value, logical basis index of the stop entry; -1 when the whole distribution weighs less than the bound).

        The stable ascending (E(k), logical k) order is the order of the composite key (energy_key(E(k)), k) -- for alpha ~ 1
        the key is k alone -- and the stop entry is the smallest key whose inclusive mass reaches alpha - isclose tolerance: a
        weighted selection.  Every pass histograms the next 8-bit digit of the key over the entries matching the prefix fixed
        so far, on every shard (``qb_cvar_select_device``); the host adds the shards' buckets in rank order and keeps the bucket
        in which the bound falls.  The energy phase ends as soon as that bucket holds one distinct energy, the select as soon
        as it holds one entry.  Logical index bits are read from their physical positions: no data moves.  The first pass
        stores (p, E) of every entry in the idle spare buffer, the later ones read it from there.  Every rank makes the same
        decisions from the same all-gathered numbers, so every caller gets the same result.  ``cache=False`` recomputes p and E
        from the state on every pass instead (same values)."""
        from . import expectation as ex
        from .engine import merge_duplicate_terms

        ex.check_alpha(alpha)
        _, zs, cs = merge_duplicate_terms(np.zeros(len(z_masks), dtype=np.uint64), np.asarray(z_masks, dtype=np.uint64), np.asarray(coeffs, dtype=np.float64))
        phys = np.asarray([self._physical_mask(z) for z in zs], dtype=np.uint64)
        cf = np.ascontiguousarray(np.real(cs), dtype=np.float64)
        bound = alpha - (1e-8 + 1e-5 * alpha)
        energy_phase = not ex._close(alpha, 1)
        e_prefix, e_free = 0, 64  # energy key bits fixed so far (64 open: no constraint)
        idx_mask = idx_value = 0  # physical index bits fixed by the logical-index prefix
        hi = self.n_qubits  # logical bits >= hi are fixed
        below_m = below_s = 0.0  # mass and sum p * E of every entry whose key is below the current prefix range
        self.cvar_passes = 0
        while True:
            if energy_phase:
                lo, spec = hi, (e_prefix, e_free, 0, (), idx_mask, idx_value)
            else:
                lo = max(0, hi - 8)
                spec = (e_prefix, e_free, 1, [self.position[q] for q in range(lo, hi)], idx_mask, idx_value)
            parts = self._select_pass(phys, cf, 0 if not cache else 1 if self.cvar_passes == 0 else 2, spec)
            self.cvar_passes += 1
            mass, pe = np.zeros(256), np.zeros(256)
            count = np.zeros(256, dtype=np.uint64)
            emin, emax, kmin = np.full(256, ~np.uint64(0)), np.zeros(256, dtype=np.uint64), np.full(256, ~np.uint64(0))
            for sums, ints in parts:  # rank order: every rank adds the same numbers in the same order
                mass, pe = mass + sums[0], pe + sums[1]
                count = count + ints[0]
                emin, emax, kmin = np.minimum(emin, ints[1]), np.maximum(emax, ints[2]), np.minimum(kmin, ints[3])
            mass_l, pe_l, count_l = mass.tolist(), pe.tolist(), count.tolist()
            before_m, before_s, run_m, run_s = [], [], below_m, below_s
            for b in range(256):
                before_m.append(run_m), before_s.append(run_s)
                run_m += mass_l[b]
                run_s += pe_l[b]
            if self.cvar_passes == 1 and run_m < bound:  # the whole distribution weighs less than the bound: every entry is taken
                return run_s / alpha, -1
            hits = [b for b in range(256) if count_l[b] and before_m[b] + mass_l[b] >= bound]
            if hits:
                pick = hits[0]
            else:  # this bucket's parent reached the bound, its digits' sums miss it by rounding only: the last entry with mass stops
                pick = ([b for b in range(256) if count_l[b] and mass_l[b] > 0] or [b for b in range(256) if count_l[b]])[-1]
            below_m, below_s = before_m[pick], before_s[pick]
            if count_l[pick] == 1:
                p, e = mass_l[pick], energy_from_key(emin[pick])
                k = int(kmin[pick])
                logical = sum(((k >> self.position[q]) & 1) << q for q in range(self.n_qubits))
                return (below_s + min(alpha - below_m, p) * e) / alpha, logical
            if energy_phase:
                if emin[pick] == emax[pick]:  # one distinct energy left: ties are ordered by the logical index
                    e_prefix, e_free, energy_phase = int(emin[pick]), 0, False
                else:
                    e_prefix, e_free = (e_prefix << 8) | pick, e_free - 8
                continue
            for j, q in enumerate(range(lo, hi)):
                idx_mask |= 1 << self.position[q]
                idx_value |= ((pick >> j) & 1) << self.position[q]
            hi = lo
            if hi == 0:
                raise RuntimeError("cvar select: the full logical index matched more than one entry")

    def sample(self, shots: int, seed=None, uniforms: Optional[np.ndarray] = None) -> np.ndarray:
        """``shots`` basis-state indices (logical qubit order) drawn from |psi|^2; every caller gets all of them.

        [upstream] Statevector.sample_memory semantics per shot (inverse-CDF of one uniform), evaluated in two levels: the
        shard masses pick the shard of every shot, the owning shard then inverts its own CDF with the re-scaled
        uniform (qb_sample_device); the physical index (rank bits | local index) is mapped back through the qubit
        permutation.  The enumeration order of the CDF is the physical one, so for given uniforms the draws are a different
        -- equally distributed -- realisation than the single-GPU sampler's unless the permutation is the identity."""
        if uniforms is None:
            uniforms = np.random.default_rng(seed).random(shots)
        u = np.ascontiguousarray(uniforms, dtype=np.float64).reshape(-1)
        masses = np.asarray(self._shard_masses(), dtype=np.float64)
        edges = np.concatenate([[0.0], np.cumsum(masses)])
        scaled = u * edges[-1]
        owner = np.minimum(np.searchsorted(edges[1:], scaled, side="right"), self.world - 1)
        with np.errstate(divide="ignore", invalid="ignore"):
            local_u = np.clip((scaled - edges[owner]) / masses[owner], 0.0, np.nextafter(1.0, 0.0))
        physical = np.asarray(self._sample_shards(owner, local_u), dtype=np.int64)
        logical = np.zeros_like(physical)
        for q in range(self.n_qubits):
            logical |= ((physical >> self.position[q]) & 1) << q
        return logical

    def describe(self) -> dict:
        return {"n_qubits": self.n_qubits, "shards": self.world, "n_local": self.n_local, "swaps_done": self.swaps_done, "swap_path": self.swap_path,
                "swap_fallback_reason": self.swap_fallback_reason}

    def _logical_from_physical(self, full: np.ndarray) -> np.ndarray:
        n = self.n_qubits
        # physical axis a <-> physical bit n-1-a ; logical bit q lives at physical position[q]
        perm = [n - 1 - self.position[q] for q in range(n - 1, -1, -1)]
        return np.ascontiguousarray(full.reshape((2,) * n).transpose(perm)).reshape(-1)


class _DeviceBuffer:
    """cudaMalloc allocation owned by an engine, usable as a torch tensor through ``__cuda_array_interface__``."""

    def __init__(self, engine, n_amplitudes: int):
        self.engine, self.size = engine, int(n_amplitudes)
        self.ptr = engine.device_alloc(16 * self.size)
        self.__cuda_array_interface__ = {"shape": (self.size,), "typestr": "<c16", "data": (self.ptr, False), "version": 3, "strides": None}

    def free(self):
        if self.ptr:
            self.engine.device_free(self.ptr)
            self.ptr = 0

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class ShardedStatevector(_ShardedLogic):
    """One process per GPU / rank; collectives over ``torch.distributed`` (NCCL on GPUs, gloo in the CPU tests)."""

    def __init__(self, n_qubits: int, backend=None, group=None, device=None, min_local: int = 12):
        import torch
        import torch.distributed as dist

        self._torch, self._dist = torch, dist
        self.group = group
        world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self._init_logic(n_qubits, world, min_local)
        if backend is None:
            from .primitives import get_engine

            dev_index = torch.cuda.current_device() if device is None else torch.device(device).index
            backend = CudaShardBackend(get_engine(dev_index, "complex128"))
            device = torch.device("cuda", dev_index)
        self.backend = backend
        self.device = torch.device("cpu") if device is None else torch.device(device)
        size = 1 << self.n_local
        self._peer_ptrs = None  # data_ptr of a local buffer -> that buffer's address on every rank, as mapped into this process
        self._owned: list = []
        self._mapped: list = []
        want_p2p = self.world > 1 and self.device.type == "cuda" and hasattr(backend, "swap_p2p") and hasattr(backend, "engine")
        if want_p2p and os.environ.get("QB_SWAP", "p2p") == "nccl":
            want_p2p, self.swap_fallback_reason = False, "QB_SWAP=nccl"
        if want_p2p:
            self._setup_ipc_buffers(size)
        if self._peer_ptrs is None:
            self.state = torch.zeros(size, dtype=torch.complex128, device=self.device)
            self.spare = torch.empty(size, dtype=torch.complex128, device=self.device)

    def _setup_ipc_buffers(self, size: int) -> None:
        """Shard buffers = cudaMalloc allocations of this rank's engine; every rank maps every other rank's buffers through
        CUDA IPC handles (all-gathered).  All ranks must agree on the outcome, so failures are all-reduced."""
        torch, dist = self._torch, self._dist
        engine = self.backend.engine
        error, bufs, handles = None, [], []
        try:
            bufs = [_DeviceBuffer(engine, size) for _ in range(2)]
            handles = [engine.ipc_export(b.ptr) for b in bufs]
        except Exception as exc:  # noqa: BLE001
            error = repr(exc)
        gathered = [None] * self.world
        dist.all_gather_object(gathered, (error, handles), group=self.group)
        failed = [e for e, _ in gathered if e]
        peer = [[0] * self.world for _ in range(2)]
        if not failed:
            try:
                for r, (_, hs) in enumerate(gathered):
                    for i in range(2):
                        if r == self.rank:
                            peer[i][r] = bufs[i].ptr
                        else:
                            peer[i][r] = engine.ipc_open(hs[i])
                            self._mapped.append(peer[i][r])
            except Exception as exc:  # noqa: BLE001
                error = repr(exc)
        flags = [None] * self.world
        dist.all_gather_object(flags, error, group=self.group)
        failed = failed or [e for e in flags if e]
        if failed:
            self.swap_fallback_reason = "no CUDA IPC peer mapping: " + failed[0]
            for p in self._mapped:
                try:
                    engine.ipc_close(p)
                except Exception:  # noqa: BLE001
                    pass
            self._mapped = []
            for b in bufs:
                b.free()
            return
        self._owned = bufs
        tensors = [torch.as_tensor(b, device=self.device) for b in bufs]
        self._peer_ptrs = {t.data_ptr(): peer[i] for i, t in enumerate(tensors)}
        self.state, self.spare = tensors
        self.state.zero_()
        torch.cuda.synchronize(self.device)
        dist.barrier(group=self.group)

    def close(self):
        """Unmap the peers' buffers and free the own ones (collective: every rank must call it before its peers free theirs)."""
        if self._peer_ptrs is not None:
            self._torch.cuda.synchronize(self.device)
            self._dist.barrier(group=self.group)
            for p in self._mapped:
                self.backend.engine.ipc_close(p)
            self._mapped = []
            self._dist.barrier(group=self.group)
            self.state = self.spare = None
            for b in self._owned:
                b.free()
            self._owned, self._peer_ptrs = [], None

    @property
    def swap_path(self) -> str:
        if self.world == 1:
            return "none (one shard)"
        return "swap_p2p_kernel over CUDA-IPC-mapped peer buffers" if self._peer_ptrs is not None else "pack + all_to_all_single + unpack"

    @property
    def index_offset(self) -> int:
        return self.rank << self.n_local

    def _apply(self, segment, params, n_params, fresh):
        self.backend.apply(self.state, segment, params, self.n_local, n_params, self.index_offset, fresh)

    def _swap(self, lp: list) -> None:
        g, nl = self.n_global, self.n_local
        torch, dist = self._torch, self._dist
        if self._peer_ptrs is not None:
            # one kernel: every amplitude goes straight to the rank that owns it afterwards, at its final index
            self.backend.swap_p2p(self.state, self._peer_ptrs[self.spare.data_ptr()], nl, self.rank, lp)
            dist.barrier(group=self.group)  # every rank's stores have landed before anyone reads its new shard
            self.state, self.spare = self.spare, self.state
            return
        # tensor axis a <-> bit nl-1-a ; bring the chosen bits to the front, most significant first = rank bit g-1
        front_bits = [lp[j] for j in range(g - 1, -1, -1)]
        rest_bits = [b for b in range(nl - 1, -1, -1) if b not in lp]
        perm = [nl - 1 - b for b in front_bits + rest_bits]
        packed = self.spare.view((2,) * nl)
        packed.copy_(self.state.view((2,) * nl).permute(perm))  # pack
        send = self.spare.view(self.world, -1)
        recv = self.state.view(self.world, -1)
        dist.all_to_all_single(recv.view(-1), send.view(-1), group=self.group)  # chunk i <-> rank i
        # received chunk j came from rank j and carries its elements with (chosen local bits) == my rank;
        # its position j now plays the role of the chosen local bits -> undo the packing permutation
        inverse = [0] * nl
        for axis, src in enumerate(perm):
            inverse[src] = axis
        self.spare.view((2,) * nl).copy_(self.state.view((2,) * nl).permute(inverse))  # unpack
        self.state, self.spare = self.spare, self.state

    def _sum_over_shards(self, fn) -> float:
        part = fn(self.backend, self.state, self.index_offset)
        if self.world == 1:
            return float(part)
        t = self._torch.tensor([part], dtype=self._torch.float64, device=self.device)
        self._dist.all_reduce(t, group=self.group)
        return float(t.item())

    def _shard_masses(self) -> np.ndarray:
        mass = self.backend.diagonal_expectation(self.state, np.zeros(1, dtype=np.uint64), np.ones(1), self.n_qubits, self.n_local, self.index_offset)
        if self.world == 1:
            return np.array([mass])
        masses = self._torch.zeros(self.world, dtype=self._torch.float64, device=self.device)
        masses[self.rank] = mass
        self._dist.all_reduce(masses, group=self.group)
        return masses.cpu().numpy()

    def _select_pass(self, z_masks, coeffs, cache_mode: int, spec) -> list:
        sums, ints = self.backend.cvar_select(self.state, self.spare, cache_mode, z_masks, coeffs, self.n_qubits, self.n_local, self.index_offset, spec)
        if self.world == 1:
            return [(sums, ints)]
        # all_gather, not all_reduce: every rank adds the shards' buckets in rank order with the same host arithmetic and so takes
        # the same bucket decision (the bits travel as int64)
        torch = self._torch
        mine = np.concatenate([np.ascontiguousarray(sums, dtype=np.float64).reshape(-1).view(np.int64),
                               np.ascontiguousarray(ints, dtype=np.uint64).reshape(-1).view(np.int64)])
        t = torch.from_numpy(mine).to(self.device)
        parts = [torch.empty_like(t) for _ in range(self.world)]
        self._dist.all_gather(parts, t, group=self.group)
        out = []
        for part in parts:
            a = part.cpu().numpy()
            out.append((a[:512].view(np.float64).reshape(2, 256), a[512:].view(np.uint64).reshape(4, 256)))
        return out

    def _sample_shards(self, owner: np.ndarray, local_u: np.ndarray) -> np.ndarray:
        physical = np.zeros(owner.size, dtype=np.int64)
        mine = np.nonzero(owner == self.rank)[0]
        if mine.size:
            physical[mine] = self.backend.sample(self.state, local_u[mine], self.n_local) | (self.rank << self.n_local)
        if self.world > 1:
            t = self._torch.from_numpy(physical).to(self.device)
            self._dist.all_reduce(t, group=self.group)  # the ranks fill disjoint shots
            physical = t.cpu().numpy()
        return physical

    def gather_physical(self) -> np.ndarray:
        """Full statevector in *physical* bit order (rank bits on top) on every rank (testing at small sizes only)."""
        torch, dist = self._torch, self._dist
        if self.world == 1:
            return self.state.cpu().numpy()
        parts = [torch.empty_like(self.state) for _ in range(self.world)]
        dist.all_gather(parts, self.state, group=self.group)
        return torch.cat(parts).cpu().numpy()

    def gather_logical(self) -> Optional[np.ndarray]:
        """Full statevector in *logical* qubit order on every rank (testing at small sizes only)."""
        return self._logical_from_physical(self.gather_physical())


class LocalShardedStatevector(_ShardedLogic):
    """ONE process, all shards: ``engines[r]`` (one per shard; the same engine may appear several times -- several shards on one
    GPU, used by the single-GPU tests) owns shard r's two buffers.  Shard-local work of all devices runs concurrently on one
    worker thread per shard (the native calls release the GIL); the swap kernel of every device stores into the other devices'
    buffers through peer access (``cudaDeviceEnablePeerAccess``); reductions happen on the host.  This is what the evaluators
    use for circuits too wide for one GPU."""

    def __init__(self, n_qubits: int, engines: Sequence, min_local: int = 12):
        from concurrent.futures import ThreadPoolExecutor

        engines = list(engines)
        self._init_logic(n_qubits, len(engines), min_local)
        self.engines = engines
        self.backends = [CudaShardBackend(e) for e in engines]
        devices = [e.device for e in engines]
        for e in engines:
            for d in set(devices):
                e.enable_peer_access(d)  # raises (with the reason) when the GPUs cannot map each other's memory
        size = 1 << self.n_local
        self._bufs = [[_DeviceBuffer(e, size) for e in engines] for _ in range(2)]  # [which][shard]
        self._cur = 0
        self._pool = ThreadPoolExecutor(max_workers=len(engines), thread_name_prefix="qb-shard") if len(engines) > 1 else None

    @property
    def swap_path(self) -> str:
        return "none (one shard)" if self.world == 1 else "swap_p2p_kernel over peer access (one process)"

    def close(self):
        for e in set(self.engines):
            e.synchronize()
        for pair in self._bufs:
            for b in pair:
                b.free()
        if self._pool is not None:
            self._pool.shutdown(wait=True)
            self._pool = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _state(self, r: int) -> int:
        return self._bufs[self._cur][r].ptr

    def _each(self, fn):
        """fn(rank) on every shard, concurrently; returns the results in shard order (first failure is raised after all ended)."""
        if self._pool is None:
            return [fn(r) for r in range(self.world)]
        futures = [self._pool.submit(fn, r) for r in range(self.world)]
        out, error = [], None
        for f in futures:
            try:
                out.append(f.result())
            except BaseException as exc:  # noqa: BLE001
                error = error or exc
                out.append(None)
        if error is not None:
            raise error
        return out

    def _apply(self, segment, params, n_params, fresh):
        self._each(lambda r: self.backends[r].apply(self._state(r), segment, params, self.n_local, n_params, r << self.n_local, fresh))

    def _swap(self, lp: list) -> None:
        dst = [self._bufs[1 - self._cur][r].ptr for r in range(self.world)]
        # every shard's kernel stores into all destination buffers; swap_p2p returns once its own stores completed, and _each
        # joins all of them: the barrier of the multi-process driver
        self._each(lambda r: self.backends[r].swap_p2p(self._state(r), dst, self.n_local, r, lp))
        self._cur = 1 - self._cur

    def _sum_over_shards(self, fn) -> float:
        return float(sum(self._each(lambda r: fn(self.backends[r], self._state(r), r << self.n_local))))

    def _shard_masses(self) -> np.ndarray:
        z, c = np.zeros(1, dtype=np.uint64), np.ones(1)
        return np.asarray(self._each(lambda r: self.backends[r].diagonal_expectation(self._state(r), z, c, self.n_qubits, self.n_local, r << self.n_local)))

    def _select_pass(self, z_masks, coeffs, cache_mode: int, spec) -> list:
        spare = self._bufs[1 - self._cur]
        return self._each(lambda r: self.backends[r].cvar_select(self._state(r), spare[r].ptr, cache_mode, z_masks, coeffs, self.n_qubits, self.n_local,
                                                                 r << self.n_local, spec))

    def _sample_shards(self, owner: np.ndarray, local_u: np.ndarray) -> np.ndarray:
        physical = np.zeros(owner.size, dtype=np.int64)

        def work(r):
            mine = np.nonzero(owner == r)[0]
            if mine.size:
                physical[mine] = self.backends[r].sample(self._state(r), local_u[mine], self.n_local) | (r << self.n_local)

        self._each(work)
        return physical

    def gather_physical(self) -> np.ndarray:
        size = 1 << self.n_local
        full = np.empty(self.world * size, dtype=np.complex128)
        for r in range(self.world):
            self.engines[r].device_read(self._state(r), 0, full[r * size : (r + 1) * size])
        return full

    def gather_logical(self) -> np.ndarray:
        return self._logical_from_physical(self.gather_physical())
