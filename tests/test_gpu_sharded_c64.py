"""Sharded statevectors in complex64 on the GPU: states and <H> against the oracle, the one-buffer route bit-identical to the
two-buffer route, every read-out equal to that read-out computed in NumPy from the state's own gathered amplitudes, the primitives
with ``dtype="complex64"`` at sharded widths, and a 34-qubit state on 2 virtual shards (64 GiB each, 64-bit indices).  One B200
runs the shards virtually (the same engine several times, as in test_gpu_sharded_local.py); with 2 and 8 GPUs the widths only
complex64 with one buffer per GPU holds (35 and 37 qubits) are checked against closed forms, and the multi-process driver against
the one-process driver."""
import math
import os

import numpy as np
import pytest

from oracle import c_oracle
from oracle import qiskit_semantics as oq
from queasars_b200 import _native
from queasars_b200 import expectation as ex
from queasars_b200 import gate_list as gl
from queasars_b200.operators import SparsePauliOp
from tests.test_gpu_cvar_exact import evqe_case
from tests.test_gpu_parity import random_ising, rel_err, tfim
from tests.test_gpu_sharded_cvar import stop_of
from tests.test_gpu_sharded_inplace import diag_of, free_or_skip, oracle_state

pytestmark = pytest.mark.gpu

GiB = 1 << 30
TOL = 1e-5


def engines64(count):
    """``count`` complex64 shards over the visible GPUs (round robin): one per GPU when there are enough, virtual shards otherwise."""
    from queasars_b200.primitives import get_engine

    n_dev = _native.device_count()
    return [get_engine(r % n_dev, "complex64") for r in range(count)]


def probs64(amps):
    return amps.real.astype(np.float64) ** 2 + amps.imag.astype(np.float64) ** 2


def chain_ising(n, seed):
    """Z on every qubit and ZZ on neighbours, random coefficients: (z masks, coefficients)."""
    rng = np.random.default_rng(seed)
    z = [1 << q for q in range(n)] + [(1 << q) | (1 << (q + 1)) for q in range(n - 1)]
    return z, [float(v) for v in rng.normal(size=len(z))]


def check_readouts(sv, z, c, energies, uniforms):
    """Every read-out of ``sv`` against NumPy on the state's own gathered amplitudes (``energies``: E(k) of sum_t c_t Z^{z_t} in
    logical order); returns them as bytes / reprs."""
    n = sv.n_qubits
    phys = sv.gather_physical()
    assert phys.dtype == np.complex64
    logical = sv.gather_logical()
    p = probs64(logical)
    out = {}
    # top states: same indices, probabilities bit for bit
    idx, tp = sv.top_states(20)
    order = np.lexsort((np.arange(p.size), -p))[:20]
    order = order[p[order] > 0]
    assert idx.tolist() == order.tolist() and tp.tobytes() == p[order].tobytes()
    out["top"] = (idx.tobytes(), tp.tobytes())
    # cvar: value within 1e-12 relative, stop entry of the stable (E, k) sort
    cv = []
    for alpha in (0.05, 0.5, 1.0):
        value, stop = sv.cvar(z, c, alpha)
        want = ex.lower_tail_expectation_arrays(p, energies, alpha)
        assert abs(value - want) <= 1e-12 * max(1.0, abs(want)), (alpha, value, want)
        assert stop == stop_of(p, energies, alpha), alpha
        cv.append((value, stop))
    out["cvar"] = repr(cv)
    # marginal on qubits that sit on rank bits and on local bits
    rank_qubits = [q for q in range(n) if sv.position[q] >= sv.n_local]
    qubits = rank_qubits[:2] + [q for q in (0, n // 2, n - 1) if q not in rank_qubits[:2]]
    m = sv.marginal(qubits)
    bins = np.zeros(p.size, dtype=np.int64)
    k = np.arange(p.size, dtype=np.int64)
    for j, q in enumerate(qubits):
        bins |= ((k >> q) & 1) << j
    assert np.max(np.abs(m - np.bincount(bins, weights=p, minlength=1 << len(qubits)))) <= 1e-12
    out["marginal"] = m.tobytes()
    # samples: the inverse CDF in physical order, mapped to logical indices; a re-scaled uniform may land on a CDF neighbour
    got = sv.sample(uniforms.size, uniforms=uniforms)
    want_phys = oq.sample_indices(phys, uniforms.size, uniforms=uniforms)
    pp = probs64(phys)
    cum = np.cumsum(pp) / pp.sum()
    got_phys = np.zeros_like(got)
    for q in range(n):
        got_phys |= ((got >> q) & 1) << sv.position[q]
    diff = np.flatnonzero(got_phys != want_phys)
    assert np.all(pp[got_phys] > 0)
    if diff.size:
        lo, hi = np.minimum(got_phys[diff], want_phys[diff]), np.maximum(got_phys[diff], want_phys[diff])
        assert np.max(cum[hi - 1] - cum[lo]) < 1e-6  # nothing with mass lies between the two draws
    assert diff.size <= max(2, uniforms.size // 1000)
    out["sample"] = got.tobytes()
    return out


@pytest.mark.parametrize("n,shards,layers", [(14, 2, 3), (17, 4, 3), (20, 8, 3), (24, 8, 2)])
def test_complex64_against_the_oracle_and_one_buffer_equals_two(n, shards, layers):
    from queasars_b200.sharded import LocalShardedStatevector

    instr, values, circ = evqe_case(n, layers, 900 + n + shards)
    gates = gl.from_circuit(circ)
    want = oracle_state(instr, n, values)
    z, c = chain_ising(n, 31 + n)
    energies = c_oracle.diag_table(n, list(zip(z, c)))
    e_diag = float(np.dot(np.abs(want) ** 2, energies))
    terms = tfim(n) + [("X" + "I" * (n - 2) + "Y", 0.3 - 0.2j)]  # X / Y on the top qubit: flips a rank bit -> one more swap
    e_tfim = oq.estimator_expectation(want, terms)
    uniforms = np.random.default_rng(n).random(10000)
    got = {}
    for buffers in (2, 1):
        sv = LocalShardedStatevector(n, engines64(shards), min_local=8, buffers=buffers)
        assert sv.dtype == sv.describe()["dtype"] == "complex64" and sv.buffers == buffers
        sv.run(gates, values)
        assert sv.swaps_done >= 1
        out = {"state": sv.gather_physical().tobytes(), "position": list(sv.position)}
        assert np.linalg.norm(sv.gather_logical() - want) <= TOL
        assert rel_err(sv.diagonal_expectation(z, c), e_diag) <= TOL
        swaps = sv.swaps_done
        assert rel_err(sv.expectation(SparsePauliOp.from_list(terms)), e_tfim) <= TOL
        assert sv.swaps_done > swaps
        assert np.linalg.norm(sv.gather_logical() - want) <= TOL
        out.update(after=(sv.gather_physical().tobytes(), list(sv.position)), **check_readouts(sv, z, c, energies, uniforms))
        got[buffers] = out
        sv.close()
    for key in got[2]:
        assert got[1][key] == got[2][key], key


@pytest.mark.parametrize("alpha", [0.2, 1.0])
def test_primitives_in_complex64_at_sharded_widths(alpha):
    """Estimator, sampler and the three evaluators with ``dtype="complex64"`` route 15-qubit circuits to a complex64 state on 4
    shards: the same values as the unsharded complex64 primitives and the oracle, and a sampled distribution within the
    total-variation bound."""
    from queasars_b200 import B200EstimatorV2, B200SamplerV2, DiagonalEnergyBitstringEvaluator
    from queasars_b200.evaluators import B200BitstringCircuitEvaluator, B200OperatorCircuitEvaluator, B200OperatorSamplerCircuitEvaluator

    n = 15
    terms = random_ising(n, 6)
    z, c = diag_of(terms)
    diag = SparsePauliOp.from_list(terms)
    energies = oq.diagonal_table(n, list(zip(z, c)))
    cases = [evqe_case(n, 3, 60 + s) for s in range(3)]
    circuits, params = [cc for _, _, cc in cases], [v for _, v, _ in cases]
    states = [oracle_state(instr, n, values) for instr, values, _ in cases]
    probs = [np.abs(s) ** 2 for s in states]
    op_terms = tfim(n) + terms[:20]
    op = SparsePauliOp.from_list(op_terms)
    est = B200EstimatorV2(devices="all", dtype="complex64", coalesce=False, shard_min_qubits=14)
    est._engines_obj = engines64(4)
    got = B200OperatorCircuitEvaluator(est, 0.0, op).evaluate_circuits(circuits, params)
    ref = B200OperatorCircuitEvaluator(B200EstimatorV2(device=0, dtype="complex64", coalesce=False), 0.0, op).evaluate_circuits(circuits, params)
    for g, r, s in zip(got, ref, states):
        assert rel_err(g, oq.estimator_expectation(s, op_terms)) <= TOL and rel_err(g, r) <= TOL
    assert est._sharded_obj[n].dtype == "complex64" and est._sharded_obj[n].world == 4
    smp = B200SamplerV2(devices="all", dtype="complex64", seed=5, coalesce=False, shard_min_qubits=14)
    smp._engines_obj = engines64(4)
    one = B200SamplerV2(device=0, dtype="complex64", coalesce=False)
    bits = DiagonalEnergyBitstringEvaluator(n, z, c)
    for kind, make in (("operator", lambda s: B200OperatorSamplerCircuitEvaluator(s, None, diag, alpha)),
                       ("bitstring", lambda s: B200BitstringCircuitEvaluator(s, None, bits, alpha))):
        for g, w, p in zip(make(smp).evaluate_circuits(circuits, params), make(one).evaluate_circuits(circuits, params), probs):
            if kind == "operator" and alpha == 1.0:  # <H> itself (the diagonal expectation of the sharded state)
                exact = float(np.dot(p, energies))
            else:
                exact = ex.lower_tail_expectation_arrays(p, energies, alpha)
            assert rel_err(g, w) <= TOL and rel_err(g, exact) <= TOL, (kind, g, w, exact)
    assert smp._sharded_obj[n].dtype == "complex64"
    shots = 20000
    idx = smp.sample_indices([circuits[0]], [params[0]], shots)[0]
    emp = np.bincount(idx, minlength=1 << n) / shots
    bound = 1.5 * 0.5 * np.sum(np.sqrt(2 * probs[0] * (1 - probs[0]) / (math.pi * shots)))
    assert 0.5 * np.abs(emp - probs[0]).sum() <= bound
    top, tp = smp.top_states([circuits[0]], [params[0]], 8)[0]
    top1, tp1 = one.top_states([circuits[0]], [params[0]], 8)[0]
    assert np.max(np.abs(tp - tp1)) <= TOL * tp1[0] and np.max(np.abs(tp - probs[0][top])) <= TOL * tp1[0]
    qs = [0, n - 1, 7]
    m = smp.marginal_probabilities([circuits[0]], [params[0]], qs)[0]
    m1 = one.marginal_probabilities([circuits[0]], [params[0]], qs)[0]
    assert np.max(np.abs(m - m1)) <= TOL


def u_product(n, theta, phi, lam, top_layers=2):
    """``u(theta, phi, lam)`` on every qubit, then ``top_layers`` more ``u`` gates on the top qubit (which start on a rank bit:
    each forces a global swap).  Product state: qubit q has p1 = sin^2(theta_q / 2) with theta_q = theta, except the top one."""
    from queasars_b200 import QuantumCircuit

    circ = QuantumCircuit(n)
    for q in range(n):
        circ.u(theta, phi, lam, q)
    for _ in range(top_layers):
        circ.u(0.35, 0.2, -0.1, n - 1)
    return circ


def u_single(theta, phi, lam):
    return np.array([[math.cos(theta / 2), -np.exp(1j * lam) * math.sin(theta / 2)],
                     [np.exp(1j * phi) * math.sin(theta / 2), np.exp(1j * (phi + lam)) * math.cos(theta / 2)]])


def product_closed_forms(n, theta, phi, lam, top_layers=2):
    """Single-qubit states of ``u_product`` -> (p1 per qubit, <X> per qubit)."""
    base = u_single(theta, phi, lam) @ np.array([1, 0])
    top = base
    for _ in range(top_layers):
        top = u_single(0.35, 0.2, -0.1) @ top
    qubit = [base] * (n - 1) + [top]
    p1 = [float(abs(v[1]) ** 2) for v in qubit]
    xs = [float(2 * (np.conj(v[0]) * v[1]).real) for v in qubit]
    return p1, xs


def check_product(sv, n, p1, xs):
    """<Ising>, <sum X>, a 3-qubit marginal with a rank-bit qubit, the top state and the norm of a product state."""
    zs = [1 - 2 * p for p in p1]
    assert abs(sv.norm_squared() - 1.0) <= TOL
    ising_z = [1 << q for q in range(n)] + [(1 << q) | (1 << (q + 1)) for q in range(n - 1)]
    ising_c = [0.5] * n + [-1.0] * (n - 1)
    want = sum(0.5 * z for z in zs) - sum(zs[q] * zs[q + 1] for q in range(n - 1))
    assert rel_err(sv.diagonal_expectation(ising_z, ising_c), want) <= TOL
    sum_x = SparsePauliOp.from_list([("I" * (n - 1 - q) + "X" + "I" * q, 1.0) for q in range(n)])
    assert rel_err(sv.expectation(sum_x), sum(xs)) <= TOL
    rank_q = [q for q in range(n) if sv.position[q] >= sv.n_local][0]
    qubits = [rank_q, 0, 5] if rank_q not in (0, 5) else [rank_q, 1, 6]
    m = sv.marginal(qubits)
    for b in range(8):
        want_b = math.prod(p1[q] if (b >> j) & 1 else 1 - p1[q] for j, q in enumerate(qubits))
        assert abs(m[b] - want_b) <= TOL * max(want_b, 1e-3), (b, m[b], want_b)
    idx, p = sv.top_states(1)
    best = sum(1 << q for q in range(n) if p1[q] > 0.5)
    assert int(idx[0]) == best
    p_best = math.prod(max(v, 1 - v) for v in p1)
    assert abs(float(p[0]) - p_best) <= TOL * p_best


def test_34_qubits_complex64_on_2_virtual_shards():
    """2 x 2^33 complex64 amplitudes = 2 x 64 GiB, the size of the widest unsharded complex64 state: 64-bit indices on the shards.
    ``buffers=None`` cannot take a second set next to the first on one GPU and falls back to one buffer (the in-place exchange)."""
    import torch

    from queasars_b200.primitives import get_engine
    from queasars_b200.sharded import LocalShardedStatevector

    n, shards = 34, 2
    need = (8 << n) + 4 * GiB
    free = torch.cuda.mem_get_info(0)[0]
    if free < need:
        pytest.skip(f"a 34-qubit complex64 state on one GPU needs {need / GiB:.0f} GiB free, {free / GiB:.1f} GiB are free")
    eng = get_engine(0, "complex64")
    sv = LocalShardedStatevector(n, [eng] * shards)
    try:
        assert sv.buffers == 1 and sv.dtype == "complex64" and sv.n_local == 33
        theta, phi, lam = 2.1, 0.4, -0.7
        sv.run(gl.from_circuit(u_product(n, theta, phi, lam)), [])
        assert sv.swaps_done >= 1
        p1, xs = product_closed_forms(n, theta, phi, lam)
        check_product(sv, n, p1, xs)
    finally:
        sv.close()


# ---------------------------------------------------------------------------------------------------- several GPUs
def test_35_qubits_complex64_on_2_gpus_through_the_primitives():
    """35 qubits in complex64 are 128 GiB per GPU on 2 GPUs: only one buffer per GPU fits, and the primitives take it."""
    from queasars_b200 import B200EstimatorV2, B200SamplerV2
    from queasars_b200.evaluators import B200OperatorCircuitEvaluator

    n_dev = _native.device_count()
    if n_dev < 2:
        pytest.skip(f"35 qubits in complex64 need 2 GPUs, {n_dev} visible")
    n = 35
    free_or_skip([0, 1], (8 << (n - 1)) + 4 * GiB, "a 35-qubit complex64 state on 2 GPUs")
    theta, phi, lam = 2.1, 0.4, -0.7
    circ = u_product(n, theta, phi, lam)
    p1, xs = product_closed_forms(n, theta, phi, lam)
    zs = [1 - 2 * p for p in p1]
    op = SparsePauliOp.from_list([("I" * (n - 1 - q) + "Z" + "I" * q, 1.0) for q in range(n)])
    est = B200EstimatorV2(devices=[0, 1], dtype="complex64", coalesce=False)
    value = B200OperatorCircuitEvaluator(est, 0.0, op).evaluate_circuits([circ], [[]])[0]
    sv = est._sharded_obj[n]
    assert sv.world == 2 and sv.buffers == 1 and sv.dtype == "complex64" and sv.swaps_done >= 1
    assert rel_err(value, sum(zs)) <= TOL
    check_product(sv, n, p1, xs)
    sv.close()
    est._sharded_obj.clear()
    smp = B200SamplerV2(devices=[0, 1], dtype="complex64", coalesce=False)
    m = smp.marginal_probabilities([circ], [[]], [n - 1, 0])[0]
    want = [(1 - p1[n - 1]) * (1 - p1[0]), p1[n - 1] * (1 - p1[0]), (1 - p1[n - 1]) * p1[0], p1[n - 1] * p1[0]]
    assert np.max(np.abs(m - want)) <= TOL
    smp._sharded_obj[n].close()
    smp._sharded_obj.clear()


def test_37_qubits_complex64_on_8_gpus_closed_form():
    """37 qubits in complex64: 128 GiB per GPU on 8 GPUs, one buffer each, n_local = 34."""
    from queasars_b200.primitives import get_engine
    from queasars_b200.sharded import LocalShardedStatevector

    n_dev = _native.device_count()
    if n_dev < 8:
        pytest.skip(f"37 qubits in complex64 need 8 GPUs, {n_dev} visible")
    n = 37
    free_or_skip(list(range(8)), (8 << (n - 3)) + 4 * GiB, "a 37-qubit complex64 state on 8 GPUs")
    sv = LocalShardedStatevector(n, [get_engine(d, "complex64") for d in range(8)])
    try:
        assert sv.buffers == 1 and sv.n_local == 34
        theta, phi, lam = 2.1, 0.4, -0.7
        sv.run(gl.from_circuit(u_product(n, theta, phi, lam, top_layers=3)), [])
        assert sv.swaps_done >= 1
        check_product(sv, n, *product_closed_forms(n, theta, phi, lam, top_layers=3))
    finally:
        sv.close()


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
        sv = ShardedStatevector(n, min_local=8, dtype="complex64")
        sv.run(gl.from_circuit(circ), values)
        got = (sv.gather_physical().tobytes(), list(sv.position), sv.swaps_done, repr(sv.diagonal_expectation(z, c)), repr(sv.cvar(z, c, 0.3)),
               sv.dtype, sv.describe()["swap_path"])
        sv.close()
        if rank == 0:
            out.put(got)
    finally:
        dist.destroy_process_group()


def test_two_process_complex64_equals_one_process_at_24_qubits():
    import socket

    import torch.multiprocessing as mp

    from queasars_b200.primitives import get_engine
    from queasars_b200.sharded import LocalShardedStatevector

    n_dev = _native.device_count()
    if n_dev < 2:
        pytest.skip(f"the multi-process driver needs 2 GPUs, {n_dev} visible")
    n = 24
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, n, out)) for r in range(2)]
    [p.start() for p in procs]
    got = out.get(timeout=600)
    [p.join(120) for p in procs]
    assert all(p.exitcode == 0 for p in procs)
    instr, values, circ = evqe_case(n, 3, 2400 + n)
    z, c = diag_of(random_ising(n, 5))
    sv = LocalShardedStatevector(n, [get_engine(d, "complex64") for d in range(2)], min_local=8)
    sv.run(gl.from_circuit(circ), values)
    want = (sv.gather_physical().tobytes(), list(sv.position), sv.swaps_done, repr(sv.diagonal_expectation(z, c)), repr(sv.cvar(z, c, 0.3)),
            sv.dtype)
    sv.close()
    assert got[5] == "complex64" and got[6].startswith("swap_")
    assert got[:6] == want
