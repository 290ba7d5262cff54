"""Sharded statevectors in complex64 on CPU: the multi-process driver over gloo (world 2 and 4, NumPy shard backend, the pack +
all-to-all exchange of complex64 tensors) against the oracle, and with NumPy stand-ins for the device: the dtype every native call
receives, the buffer sizes, the uncached CVaR select of a two-buffer complex64 state, mixed engine dtypes, and a complex64
primitive at a sharded width."""
import os

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import evqe_genome as og
from oracle import qiskit_semantics as oq
from queasars_b200 import gate_list as gl
from queasars_b200 import primitives as pr
from queasars_b200.operators import SparsePauliOp
from tests.test_frontend_planner import build_circuit
from tests.test_sharded_cvar_host import ALPHAS, random_ising_masks
from tests.test_sharded_gloo import NumpyShardBackend, _free_port
from tests.test_sharded_inplace_host import MEMORY, FakeEngine, PointerBackend


# ---------------------------------------------------------------------------------------------------- multi-process driver over gloo
def _worker(rank, world, port, n, layers, seed, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from queasars_b200.sharded import ShardedStatevector

        genome, values = og.random_individual(n, layers, True, seed)
        instr = og.individual_circuit(genome, values)
        sv = ShardedStatevector(n, backend=NumpyShardBackend(), min_local=4, dtype="complex64")
        sv.run(gl.from_circuit(build_circuit(instr, n)), values)
        want = oq.statevector(instr, n, values)
        got = sv.gather_logical()
        rng = np.random.default_rng(5)
        z_masks = [int(rng.integers(0, 1 << n)) for _ in range(6)]
        coeffs = [float(c) for c in rng.normal(size=6)]
        e_got = sv.diagonal_expectation(z_masks, coeffs)
        e_want = float(np.dot(np.abs(want) ** 2, oq.diagonal_table(n, list(zip(z_masks, coeffs)))))
        labels = [("I" * (n - 1 - q) + ("X" if q % 2 else "Y") + "I" * q, float(rng.normal())) for q in range(n)] + [("Z" * n, 0.25)]
        p_got = sv.expectation(SparsePauliOp.from_list(labels))  # X / Y on rank bits: more swaps
        p_want = oq.estimator_expectation(want, labels)
        after = sv.gather_logical()
        if rank == 0:
            out.put((sv.dtype, str(sv.state.dtype), str(got.dtype), sv.describe()["dtype"], float(np.linalg.norm(got - want)),
                     float(np.linalg.norm(after - want)), abs(e_got - e_want) / max(1.0, abs(e_want)),
                     abs(p_got - p_want) / max(1.0, abs(p_want)), sv.swaps_done, sv.bytes_sent, sv.n_local))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,n,layers,seed", [(2, 8, 4, 0), (4, 9, 5, 1), (2, 10, 3, 2), (4, 10, 4, 3)])
def test_gloo_complex64_matches_oracle(world, n, layers, seed):
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, n, layers, seed, out)) for r in range(world)]
    [p.start() for p in procs]
    [p.join(120) for p in procs]
    assert all(p.exitcode == 0 for p in procs)
    dtype, tensor_dtype, gathered, described, err, err_after, e_err, p_err, swaps, sent, nl = out.get(timeout=10)
    assert dtype == described == gathered == "complex64" and tensor_dtype == "torch.complex64"
    assert err <= 1e-5 and err_after <= 1e-5 and e_err <= 1e-5 and p_err <= 1e-5
    assert swaps >= 1
    assert sent == swaps * (world - 1) * ((1 << nl) // world) * 8  # 8 bytes per amplitude


# ---------------------------------------------------------------------------------------------------- NumPy stand-ins for the device
class Engine64(FakeEngine):
    """``FakeEngine`` of test_sharded_inplace_host.py with a dtype: device memory of that dtype, every allocation's size kept."""

    def __init__(self, device=0, dtype="complex64", **kw):
        super().__init__(device, **kw)
        self.dtype, self.alloc_bytes = dtype, []

    def device_alloc(self, nbytes):
        ptr = super().device_alloc(nbytes)
        self.alloc_bytes.append(nbytes)
        MEMORY[ptr] = np.zeros(nbytes // np.dtype(self.dtype).itemsize, dtype=self.dtype)
        return ptr

    def device_read(self, ptr, offset, out):
        size = np.dtype(self.dtype).itemsize
        out[:] = MEMORY[ptr][offset // size : offset // size + out.size]
        return out


def local_state64(n, world, buffers, dtype="complex64"):
    from queasars_b200.sharded import LocalShardedStatevector

    engines = [Engine64(r, dtype) for r in range(world)]
    sv = LocalShardedStatevector(n, engines, min_local=3, buffers=buffers)
    sv.backends = [PointerBackend() for _ in range(world)]
    return sv, engines


@pytest.mark.parametrize("buffers", [2, 1])
def test_buffers_hold_8_bytes_per_amplitude(buffers):
    n, world = 9, 4
    sv, engines = local_state64(n, world, buffers)
    assert sv.dtype == sv.describe()["dtype"] == "complex64" and sv.amp_bytes == 8 and sv.buffers == buffers
    assert all(e.alloc_bytes == [8 << sv.n_local] * buffers for e in engines)
    assert all(b.__cuda_array_interface__["typestr"] == "<c8" and b.size == 1 << sv.n_local for s in sv._bufs for b in s)
    genome, values = og.random_individual(n, 4, True, 11)
    instr = og.individual_circuit(genome, values)
    sv.run(gl.from_circuit(build_circuit(instr, n)), values)
    assert sv.swaps_done >= 1 and sv.bytes_sent == sv.swaps_done * (world - 1) * ((1 << sv.n_local) // world) * 8
    got = sv.gather_logical()
    assert got.dtype == np.complex64 and sv.gather_physical().dtype == np.complex64
    assert np.linalg.norm(got - oq.statevector(instr, n, values)) <= 1e-5
    sv.close()


def test_two_buffer_complex64_cvar_runs_uncached_with_the_same_values():
    """The (p, E) cache takes 16 bytes per entry, a complex64 spare holds 8: a two-buffer complex64 state never asks for cache
    modes 1 or 2, and its values are the ones of the one-buffer state."""
    n, world = 9, 4
    genome, values = og.random_individual(n, 5, True, 21)
    gates = gl.from_circuit(build_circuit(og.individual_circuit(genome, values), n))
    z, c = random_ising_masks(n, 77)
    got = {}
    for buffers in (2, 1):
        sv, _ = local_state64(n, world, buffers)
        sv.run(gates, values)
        got[buffers] = [sv.gather_physical().tobytes()] + [sv.cvar(z, c, a) for a in ALPHAS]
        calls = [call for b in sv.backends for call in b.select_calls]
        assert calls and all(mode == 0 for _, mode in calls)
        sv.close()
    assert repr(got[1]) == repr(got[2])
    sv, _ = local_state64(n, world, 2, "complex128")  # (complex128 keeps its cache)
    sv.run(gates, values)
    sv.cvar(z, c, 0.5)
    assert {mode for b in sv.backends for _, mode in b.select_calls} == {1, 2}
    sv.close()


def test_engines_of_mixed_dtypes_raise():
    from queasars_b200.sharded import LocalShardedStatevector, ShardedStatevector

    with pytest.raises(ValueError, match="one dtype"):
        LocalShardedStatevector(8, [Engine64(0, "complex64"), Engine64(1, "complex128")], min_local=3)
    backend = type("B", (), {"engine": Engine64(0, "complex128")})()
    with pytest.raises(ValueError, match="complex64 sharded statevector"):
        ShardedStatevector(8, backend=backend, min_local=4, dtype="complex64")
    with pytest.raises(ValueError):
        ShardedStatevector(8, backend=NumpyShardBackend(), min_local=4, dtype="float64")


class RecordingEngine:
    """Records the dtype of every call of the engine's device-pointer API and returns outputs of the right shape."""

    def __init__(self, dtype):
        self.dtype, self.calls = dtype, []

    def compile(self, gates, dtype=None, from_zero_state=True):
        self.calls.append(("compile", self.dtype if dtype is None else dtype))
        return object()

    def apply_plan_device(self, plan, params, state_ptr, init_zero, index_offset):
        self.calls.append(("apply_plan_device", None))

    def hamiltonian(self, op, build_table=None):
        return object()

    def synchronize(self):
        pass

    def expectation_device(self, ham, dtype, *args):
        self.calls.append(("expectation_device", dtype))
        return 0.0

    def sample_device(self, dtype, n_local, state_ptr, uniforms):
        self.calls.append(("sample_device", dtype))
        return np.zeros(len(uniforms), dtype=np.int64)

    def cvar_select_device(self, ham, dtype, *args):
        self.calls.append(("cvar_select_device", dtype))
        return np.zeros((2, 256)), np.zeros((4, 256), dtype=np.uint64)

    def top_select_device(self, dtype, *args):
        self.calls.append(("top_select_device", dtype))
        return np.zeros(256, dtype=np.uint64)

    def top_collect_device(self, dtype, *args):
        self.calls.append(("top_collect_device", dtype))
        return np.zeros(0, dtype=np.int64), np.zeros(0)

    def marginal_device(self, dtype, n_local, state_ptr, index_offset, positions):
        self.calls.append(("marginal_device", dtype))
        return np.zeros(1 << len(positions))

    def swap_global_p2p(self, dtype, *args):
        self.calls.append(("swap_global_p2p", dtype))

    def swap_global_inplace_p2p(self, dtype, *args):
        self.calls.append(("swap_global_inplace_p2p", dtype))


@pytest.mark.parametrize("dtype", ["complex64", "complex128"])
def test_every_native_call_receives_the_engines_dtype(dtype):
    from queasars_b200.sharded import CudaShardBackend

    eng = RecordingEngine(dtype)
    b = CudaShardBackend(eng)
    z, c = np.array([1, 3], dtype=np.uint64), np.array([0.5, -1.0])
    b.apply(1 << 20, [], np.zeros(0), 10, 0, 0, True)
    b.diagonal_expectation(1 << 20, z, c, 11, 10, 0)
    b.pauli_expectation(1 << 20, [1], [2], [1.0], 11, 10, 0)
    b.sample(1 << 20, np.array([0.5]), 10)
    b.cvar_select(1 << 20, None, 0, z, c, 11, 10, 0, (0, 64, 0, (), 0, 0))
    b.top_select(1 << 20, 10, 0, 0.0, None, [0])
    b.top_collect(1 << 20, 10, 0, 0.0, None, [0], 1)
    b.marginal(1 << 20, 10, 0, [0, 10])
    b.swap_p2p(1 << 20, [1 << 21, 1 << 22], 10, 0, [9])
    b.swap_inplace_p2p(1 << 20, [1 << 20, 1 << 22], 10, 0, [9])
    names = {name for name, _ in eng.calls}
    assert names >= {"compile", "expectation_device", "sample_device", "cvar_select_device", "top_select_device", "top_collect_device",
                     "marginal_device", "swap_global_p2p", "swap_global_inplace_p2p"}
    assert all(d == dtype for name, d in eng.calls if name != "apply_plan_device")


def test_complex64_primitive_builds_its_sharded_state(monkeypatch):
    """A complex64 estimator at a sharded width builds a complex64 sharded state from its device set (no NotImplementedError), and
    its values come from that state."""
    from queasars_b200 import B200EstimatorV2
    from queasars_b200.evaluators import B200OperatorCircuitEvaluator

    monkeypatch.setattr(pr._native, "device_count", lambda: 2)
    n = 9
    est = B200EstimatorV2(devices="all", dtype="complex64", shard_min_qubits=n, coalesce=False)
    est._engines_obj = [Engine64(d, "complex64") for d in range(2)]
    sv = est._sharded_state(n)
    assert sv.dtype == "complex64" and sv.world == 2 and sv.buffers == 2
    assert all(e.alloc_bytes == [8 << (n - 1)] * 2 for e in est._engines_obj)
    sv.backends = [PointerBackend() for _ in range(2)]
    genome, values = og.random_individual(n, 4, True, 31)
    instr = og.individual_circuit(genome, values)
    terms = [("I" * (n - 1 - q) + "Z" + "I" * q, 0.5 + q) for q in range(n)] + [("X" + "I" * (n - 2) + "Z", 0.7)]
    op = SparsePauliOp.from_list(terms)
    got = B200OperatorCircuitEvaluator(est, 0.0, op).evaluate_circuits([build_circuit(instr, n)], [list(values)])[0]
    want = oq.estimator_expectation(oq.statevector(instr, n, values), terms)
    assert est._sharded_obj[n] is sv and sv.swaps_done >= 1
    assert abs(got - want) <= 1e-5 * max(1.0, abs(want))
    sv.close()
