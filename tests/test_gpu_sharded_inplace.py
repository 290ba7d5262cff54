"""Sharded statevectors with ONE buffer per shard (``swap_inplace_p2p_kernel``, the in-place global <-> local exchange) on the GPU:
bit-identical to the two-buffer route (``swap_p2p_kernel``) in states, placements and every read-out, against the oracle, the
C-ABI kernel against the NumPy permutation in both dtypes and its argument checks.  One B200 runs the shards virtually (the same
engine several times, as in test_gpu_sharded_local.py); with 2 and 8 GPUs the widths that only one buffer per GPU holds (34 and
36 qubits) are checked against closed forms, and the multi-process driver against its two-buffer route."""
import math
import os

import numpy as np
import pytest

from oracle import c_oracle
from queasars_b200 import _native
from queasars_b200 import gate_list as gl
from queasars_b200.operators import SparsePauliOp
from tests.test_gpu_cvar_exact import evqe_case
from tests.test_gpu_parity import random_ising, tfim
from tests.test_gpu_sharded_local import shard_engines
from tests.test_sharded_inplace_host import swapped_permutation

pytestmark = pytest.mark.gpu

GiB = 1 << 30


def oracle_state(instr, n, values):
    _, state = c_oracle.evaluate(instr, n, values, None, np.empty(1 << n, dtype=np.complex128))
    return state


def diag_of(terms):
    from oracle import qiskit_semantics as oq

    d = oq.diag_terms_from_labels(terms)
    return [z for z, _ in d], [c for _, c in d]


def readouts(sv, z, c, op, uniforms):
    """Everything a sharded state gives out, as bytes / reprs that compare bit for bit."""
    out = {"state": sv.gather_physical().tobytes(), "position": list(sv.position), "swaps": sv.swaps_done}
    out["diag"] = repr(sv.diagonal_expectation(z, c))
    out["pauli"] = repr(sv.expectation(op))  # X on the top qubit: one more swap inside
    out["after_pauli"] = (sv.gather_physical().tobytes(), list(sv.position), sv.swaps_done)
    out["sample"] = sv.sample(uniforms.size, uniforms=uniforms).tobytes()
    out["cvar"] = repr([sv.cvar(z, c, a) for a in (0.05, 0.5, 1.0)])
    idx, p = sv.top_states(20)
    out["top"] = (idx.tobytes(), p.tobytes())
    return out


@pytest.mark.parametrize("n,shards,layers", [(14, 2, 3), (17, 4, 3), (20, 8, 3), (24, 16, 2)])
def test_one_buffer_is_bit_identical_to_two_buffers(n, shards, layers):
    from queasars_b200.sharded import LocalShardedStatevector

    instr, values, circ = evqe_case(n, layers, 700 + n)
    gates = gl.from_circuit(circ)
    engines = shard_engines(shards)
    terms = random_ising(n, 31 + n)
    z, c = diag_of(terms)
    op = SparsePauliOp.from_list(tfim(n) + [("X" + "I" * (n - 2) + "Y", 0.3 - 0.2j)])
    uniforms = np.random.default_rng(n).random(10000)
    want = oracle_state(instr, n, values)
    got = {}
    for buffers in (2, 1):
        sv = LocalShardedStatevector(n, engines, min_local=8, buffers=buffers)
        assert sv.buffers == buffers and sv.describe()["buffers"] == buffers
        sv.run(gates, values)
        assert sv.swaps_done >= 1
        assert np.max(np.abs(sv.gather_logical() - want)) < 1e-12
        got[buffers] = readouts(sv, z, c, op, uniforms)
        assert got[buffers]["after_pauli"][2] > got[buffers]["swaps"]
        sv.close()
    assert got[1]["state"] == got[2]["state"]  # the exchange moves amplitudes, it computes nothing
    for key in got[2]:
        assert got[1][key] == got[2][key], key


@pytest.mark.parametrize("dtype", ["complex128", "complex64"])
@pytest.mark.parametrize("n_local,lp", [(2, [0]), (12, [11]), (13, [0, 12]), (3, [0, 2]), (14, [0, 5, 13]), (12, [2, 3, 4]),
                                        (5, [0, 1, 2, 4]), (15, [1, 2, 3, 14])])
def test_c_abi_exchange_is_the_bit_permutation(dtype, n_local, lp):
    """qb_swap_global_inplace_p2p with every "rank" on one GPU, on raw device buffers: each rank's kernel swaps its pairs with the
    other ranks' buffers; afterwards the buffers hold the permutation rank bit j <-> lp[j], bit for bit."""
    import torch

    from queasars_b200.primitives import get_engine

    engine = get_engine(0)
    g = len(lp)
    world = 1 << g
    rng = np.random.default_rng(n_local * 16 + g)
    full = (rng.normal(size=world << n_local) + 1j * rng.normal(size=world << n_local)).astype(dtype)
    shards = [torch.from_numpy(full[r << n_local : (r + 1) << n_local].copy()).cuda() for r in range(world)]
    torch.cuda.synchronize()
    ptrs = [s.data_ptr() for s in shards]
    for r in range(world):
        engine.swap_global_inplace_p2p(dtype, n_local, ptrs, r, lp)
    engine.synchronize()
    got = np.concatenate([s.cpu().numpy() for s in shards])
    assert got.tobytes() == swapped_permutation(full, n_local, lp).tobytes()


def test_c_abi_refuses_bad_arguments_without_launching():
    import torch

    from queasars_b200.primitives import get_engine

    engine = get_engine(0)
    bufs = [torch.zeros(1 << 10, dtype=torch.complex128, device="cuda") for _ in range(4)]
    ptrs = [b.data_ptr() for b in bufs]
    torch.cuda.synchronize()
    cases = [
        (10, ptrs, 0, [5, 2]),  # unsorted positions
        (10, ptrs, 0, [3, 3]),  # duplicate positions
        (10, ptrs[:3], 0, [2, 3]),  # world 3 != 2^2
        (10, ptrs, 0, [2, 3, 4]),  # world 4 != 2^3
        (10, ptrs[:3] + [0], 1, [2, 3]),  # a null shard buffer
        (2, ptrs, 0, [0, 1]),  # n_local < g + 1
        (10, ptrs, 0, [2, 10]),  # a position outside the shard
    ]
    for n_local, p, rank, lp in cases:
        before = engine.launch_count
        with pytest.raises(_native.QbError) as info:
            engine.swap_global_inplace_p2p("complex128", n_local, p, rank, lp)
        assert info.value.code == _native.QB_ERR_INVALID, (n_local, rank, lp)
        assert engine.launch_count == before
    engine.swap_global_inplace_p2p("complex128", 3, ptrs, 0, [0, 2])  # the smallest shard the kernel takes, g = 2
    engine.synchronize()


# ---------------------------------------------------------------------------------------------------- several GPUs
def free_or_skip(devices, need, what):
    import torch

    free = [torch.cuda.mem_get_info(d)[0] for d in devices]
    if min(free) < need:
        pytest.skip(f"{what}: needs {need / GiB:.1f} GiB free per GPU, the GPUs have {[round(f / GiB, 1) for f in free]} GiB free")


def product_circuit(n, theta, layers=1):
    from queasars_b200 import QuantumCircuit

    circ = QuantumCircuit(n)
    for _ in range(layers):
        for q in range(n):
            circ.ry(theta / layers, q)
    return circ


def closed_form_cvar(n, theta, alpha):
    """Lower tail of H = sum_q Z_q on RY(theta)^n |0>: E = n - 2 j on the C(n, j) states with j ones, p = s^j (1 - s)^(n - j);
    returns (value filled exactly to the stop bound, slack |E| p_max / alpha of the greedy fill)."""
    s = math.sin(theta / 2) ** 2
    levels = [(n - 2 * j, math.comb(n, j), s**j * (1 - s) ** (n - j)) for j in range(n, -1, -1)]
    bound = alpha - (1e-8 + 1e-5 * alpha)
    acc = taken = 0.0
    for e, cnt, p in levels:
        take = min(cnt * p, bound - taken)
        acc, taken = acc + take * e, taken + take
        if taken >= bound:
            break
    return acc / alpha, n * max(p for _, _, p in levels) / alpha + 1e-9 * n


def _nccl_worker(rank, world, port, n, out):
    import torch
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from queasars_b200.sharded import ShardedStatevector

        instr, values, circ = evqe_case(n, 3, 2400 + n)
        z, c = diag_of(random_ising(n, 5))
        got = {}
        for buffers in (2, 1):
            sv = ShardedStatevector(n, buffers=buffers, min_local=8)
            sv.run(gl.from_circuit(circ), values)
            got[buffers] = (sv.gather_physical().tobytes(), list(sv.position), sv.swaps_done, repr(sv.diagonal_expectation(z, c)),
                            repr(sv.cvar(z, c, 0.3)), sv.describe()["swap_path"], sv.buffers)
            sv.close()
        if rank == 0:
            out.put((got[1][:5] == got[2][:5], got[2][2], got[1][5], got[2][5], got[1][6]))
    finally:
        dist.destroy_process_group()


def test_two_process_one_buffer_equals_two_buffers_at_24_qubits():
    import socket

    import torch.multiprocessing as mp

    n_dev = _native.device_count()
    if n_dev < 2:
        pytest.skip(f"the multi-process driver needs 2 GPUs, {n_dev} visible")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, 24, out)) for r in range(2)]
    [p.start() for p in procs]
    same, swaps, path1, path2, buffers1 = out.get(timeout=600)
    [p.join(120) for p in procs]
    assert all(p.exitcode == 0 for p in procs)
    assert swaps >= 1 and buffers1 == 1
    assert path1.startswith("swap_inplace_p2p_kernel") and path2.startswith("swap_p2p_kernel")
    assert same


def test_34_qubits_on_2_gpus_through_the_primitives():
    """34 qubits in complex128 are 128 GiB per GPU on 2 GPUs: only one buffer per GPU fits, and the primitives take it."""
    from queasars_b200 import B200EstimatorV2, B200SamplerV2
    from queasars_b200.evaluators import B200OperatorCircuitEvaluator

    n_dev = _native.device_count()
    if n_dev < 2:
        pytest.skip(f"34 qubits need 2 GPUs, {n_dev} visible")
    n, theta = 34, 1.9
    free_or_skip([0, 1], (16 << (n - 1)) + 4 * GiB, "a 34-qubit state on 2 GPUs")
    op = SparsePauliOp.from_list([("I" * (n - 1 - q) + "Z" + "I" * q, 1.0) for q in range(n)])
    circ = product_circuit(n, theta)
    est = B200EstimatorV2(devices=[0, 1], coalesce=False)
    value = B200OperatorCircuitEvaluator(est, 0.0, op).evaluate_circuits([circ], [[]])[0]
    sv = est._sharded_obj[n]
    assert sv.world == 2 and sv.buffers == 1 and sv.swaps_done >= 1
    assert abs(value - n * math.cos(theta)) < 1e-9
    sv.close()
    est._sharded_obj.clear()
    smp = B200SamplerV2(devices=[0, 1], coalesce=False)
    for alpha in (0.05, 0.5):
        got = smp.cvar_values([circ], [[]], op, alpha)[0]
        want, slack = closed_form_cvar(n, theta, alpha)
        assert abs(got - want) <= slack, (alpha, got, want)
    assert smp._sharded_obj[n].buffers == 1
    smp._sharded_obj[n].close()
    smp._sharded_obj.clear()


def test_36_qubits_on_8_gpus_closed_form():
    """36 qubits in complex128: 128 GiB per GPU on 8 GPUs, one buffer each.  Product state RY(theta)^n: <sum Z> = n cos(theta),
    CVaR against the closed form, the most probable states; then a circuit whose gates target rank bits again and again keeps the
    norm."""
    from queasars_b200.primitives import get_engine
    from queasars_b200.sharded import LocalShardedStatevector

    n_dev = _native.device_count()
    if n_dev < 8:
        pytest.skip(f"36 qubits need 8 GPUs, {n_dev} visible")
    n, theta = 36, 1.9
    free_or_skip(list(range(8)), (16 << (n - 3)) + 4 * GiB, "a 36-qubit state on 8 GPUs")
    sv = LocalShardedStatevector(n, [get_engine(d) for d in range(8)])
    try:
        assert sv.buffers == 1
        sv.run(gl.from_circuit(product_circuit(n, theta)), [])
        z, c = [1 << q for q in range(n)], [1.0] * n
        assert abs(sv.diagonal_expectation(z, c) - n * math.cos(theta)) < 1e-9
        for alpha in (0.05, 0.5, 0.9):
            value, _ = sv.cvar(z, c, alpha)
            want, slack = closed_form_cvar(n, theta, alpha)
            assert abs(value - want) <= slack, (alpha, value, want)
        s = math.sin(theta / 2) ** 2  # > 1/2: all ones first, then the n states with one zero
        idx, p = sv.top_states(1 + n)
        ones = (1 << n) - 1
        # (the n one-zero states tie up to the rounding of their products: compared as a set)
        assert idx[0] == ones and sorted(idx[1:].tolist()) == sorted(ones ^ (1 << q) for q in range(n))
        assert np.allclose(p, [s**n] + [s ** (n - 1) * (1 - s)] * n, rtol=1e-12, atol=0) and np.all(np.diff(p) <= 0)
        sv.reset()
        swaps = sv.swaps_done
        sv.run(gl.from_circuit(product_circuit(n, 2.3, layers=3)), [])
        assert sv.swaps_done - swaps >= 2
        assert abs(sv.norm_squared() - 1.0) < 1e-12
        assert abs(sv.diagonal_expectation(z, c) - n * math.cos(2.3)) < 1e-9
    finally:
        sv.close()
