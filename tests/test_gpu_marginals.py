"""Exact marginal probabilities on the device (``qb_marginal_probabilities`` / ``Engine.marginal_probabilities``, the sharded
``_ShardedLogic.marginal`` through ``qb_marginal_device``, ``B200SamplerV2.marginal_probabilities``) against a NumPy marginal of
the same amplitudes read back with ``Engine.statevector``, and the per-register read-out of ``B200SamplerV2.run`` on the GPU."""
import math

import numpy as np
import pytest

from oracle import evqe_genome as og
from queasars_b200 import ClassicalRegister, QuantumCircuit
from queasars_b200 import gate_list as gl
from tests.test_frontend_planner import build_circuit
from tests.test_gpu_wide_states import fit_or_skip

pytestmark = pytest.mark.gpu

GiB = 1 << 30
TOL = {"complex128": 1e-13, "complex64": 1e-6}


@pytest.fixture(scope="module")
def engines():
    from queasars_b200.engine import Engine

    made = {d: Engine(device=0, dtype=d) for d in ("complex128", "complex64")}
    yield made
    for e in made.values():
        e.close()


def evqe_case(n, layers, seed):
    genome, values = og.random_individual(n, layers, True, seed)
    instr = og.individual_circuit(genome, values)
    return instr, list(values), build_circuit(instr, n)


def np_marginal(p, n, qubits):
    """Statevector.probabilities(qargs) of the probabilities p: bit j of the output index = qubit qubits[j]."""
    t = p.reshape((2,) * n)  # axis a <-> qubit n - 1 - a
    drop = tuple(n - 1 - q for q in range(n) if q not in qubits)
    t = t.sum(axis=drop) if drop else t
    kept = sorted(qubits, reverse=True)  # remaining axes, most significant qubit first
    perm = [kept.index(qubits[j]) for j in range(len(qubits) - 1, -1, -1)]
    return np.ascontiguousarray(t.transpose(perm)).reshape(-1)


def subsets(n, seed):
    rng = np.random.default_rng(seed)
    out = {"m=1 low": [0], "m=1 high": [n - 1], "m=n": list(range(n)), "low": list(range(min(8, n))), "high": list(range(n - 8, n)),
           "tile boundary": [q for q in (8, 9, 10, 11, 12, 13) if q < n], "reversed": list(range(n - 1, -1, -1))}
    for k in (3, 7, n // 2, n - 1):
        out[f"random {k}"] = [int(q) for q in rng.permutation(n)[:k]]
    return out


@pytest.mark.parametrize("dtype", ["complex128", "complex64"])
@pytest.mark.parametrize("n", [10, 16, 20])
def test_random_circuits_against_numpy(engines, dtype, n):
    eng = engines[dtype]
    _, values, circ = evqe_case(n, 4, 300 + n)
    plan = eng.compile(gl.from_circuit(circ))
    amps = eng.statevector(plan, values)
    p = amps.real * amps.real + amps.imag * amps.imag
    for what, qubits in subsets(n, n).items():
        got = eng.marginal_probabilities([plan], [values], qubits)
        assert got.shape == (1, 1 << len(qubits)) and got.dtype == np.float64
        want = np_marginal(p, n, qubits)
        assert np.max(np.abs(got[0] - want)) <= TOL[dtype], f"{dtype} n={n} {what}"
        if what == "m=n":  # every qubit measured in order: |psi|^2 itself, rounded like NumPy's re * re + im * im
            assert np.array_equal(got[0].view(np.uint64), p.view(np.uint64))
        again = eng.marginal_probabilities([plan], [values], qubits)
        assert np.array_equal(again.view(np.uint64), got.view(np.uint64)), f"{dtype} n={n} {what}: two calls differ"


def test_batch_rows_in_submission_order(engines):
    eng = engines["complex128"]
    n = 14
    cases = [evqe_case(n, 3, 40 + i) for i in range(5)]
    plans = [eng.compile(gl.from_circuit(c)) for _, _, c in cases]
    values = [v for _, v, _ in cases]
    qubits = [13, 2, 7, 0]
    got = eng.marginal_probabilities(plans + plans[:2], values + values[:2], qubits)
    assert got.shape == (7, 16)
    for i, (plan, vals) in enumerate(zip(plans + plans[:2], values + values[:2])):
        amps = eng.statevector(plan, vals)
        assert np.max(np.abs(got[i] - np_marginal(np.abs(amps) ** 2, n, qubits))) <= 1e-13, f"row {i}"


def test_validation(engines):
    from queasars_b200 import _native

    eng = engines["complex128"]
    _, values, circ = evqe_case(10, 2, 1)
    plan = eng.compile(gl.from_circuit(circ))
    for bad in ([], list(range(10)) + [0], [10], [-1], [3, 3]):
        with pytest.raises(ValueError):
            eng.marginal_probabilities([plan], [values], bad)
    # the native checks behind them
    ids, flat, offsets = eng._pack([plan], [values])
    out = np.empty(1 << 10)  # (every call below is refused before anything is written)
    for qubits in ([3, 3], [10], list(range(27))):
        q = np.asarray(qubits, dtype=np.int32)
        code = eng._lib.qb_marginal_probabilities(eng._ctx, 1, _native.ptr(ids), _native.ptr(flat), _native.ptr(offsets), q.size, _native.ptr(q), _native.ptr(out))
        assert code == _native.QB_ERR_INVALID, qubits
    buf = eng.device_alloc(16 << 10)
    try:
        with pytest.raises(_native.QbError, match="index_offset"):
            eng.marginal_device("complex128", 10, buf, 1 << 3, [0])
        with pytest.raises(_native.QbError):
            eng.marginal_device("complex128", 10, buf, 0, [0, 0])
    finally:
        eng.device_free(buf)


def test_26_of_28_qubits():
    from queasars_b200.engine import Engine

    n = 28
    fit_or_skip((16 << n) + (8 << 26) + GiB, "a 28-qubit complex128 state and a 26-qubit marginal")
    _, values, circ = evqe_case(n, 2, 28)
    eng = Engine(device=0)
    try:
        plan = eng.compile(gl.from_circuit(circ))
        amps = eng.statevector(plan, values)
        p = amps.real * amps.real + amps.imag * amps.imag
        del amps
        qubits = [int(q) for q in np.random.default_rng(28).permutation(n)[:26]]
        got = eng.marginal_probabilities([plan], [values], qubits)[0]
        assert abs(got.sum() - 1.0) < 1e-12
        assert np.max(np.abs(got - np_marginal(p, n, qubits))) <= 1e-13
        low = eng.marginal_probabilities([plan], [values], list(range(26)))[0]
        assert np.max(np.abs(low - np_marginal(p, n, list(range(26))))) <= 1e-13
    finally:
        eng.close()


def test_33_qubits_closed_form_on_64_bit_indices():
    """2^33 complex64 amplitudes: RY on qubits 0, 5, 31 and 32, H on qubit 20, |0> elsewhere; marginals of the product state."""
    from queasars_b200.engine import Engine

    n = 33
    fit_or_skip((8 << n) + 2 * GiB, "a 33-qubit complex64 state")
    thetas = {0: 0.6, 5: 1.0, 31: 2.2, 32: 1.3}
    circ = QuantumCircuit(n)
    for q, t in thetas.items():
        circ.ry(t, q)
    circ.h(20)

    def p_one(q):
        return math.sin(thetas[q] / 2) ** 2 if q in thetas else (0.5 if q == 20 else 0.0)

    eng = Engine(device=0, dtype="complex64")
    try:
        plan = eng.compile(gl.from_circuit(circ))
        for qubits in ([32], [32, 0, 31, 20, 7], [31, 32], list(range(33 - 20, 33)), [20, 5, 3, 32, 30, 0]):
            got = eng.marginal_probabilities([plan], [[]], qubits)[0]
            want = np.ones(1 << len(qubits))
            for j, q in enumerate(qubits):
                bit = (np.arange(want.size) >> j) & 1
                want *= np.where(bit == 1, p_one(q), 1.0 - p_one(q))
            assert abs(got.sum() - 1.0) < 1e-6, qubits
            assert np.allclose(got, want, rtol=2e-6, atol=1e-7), qubits
    finally:
        eng.close()


@pytest.mark.parametrize("buffers", [1, 2])
@pytest.mark.parametrize("shards", [2, 4])
def test_sharded_matches_one_gpu(shards, buffers):
    from queasars_b200.primitives import get_engine
    from queasars_b200.sharded import LocalShardedStatevector

    n = 16
    _, values, circ = evqe_case(n, 4, 700 + shards)
    gates = gl.from_circuit(circ)
    eng = get_engine(0)
    plan = eng.compile(gates)
    sv = LocalShardedStatevector(n, [eng] * shards, min_local=8, buffers=buffers)
    try:
        sv.run(gates, values)
        assert sv.swaps_done and sv.position != list(range(n))  # a global swap permuted the layout
        rank_qubits = [q for q in range(n) if sv.position[q] >= sv.n_local]
        assert rank_qubits
        cases = dict(subsets(n, shards))
        cases["rank bits"] = rank_qubits
        cases["rank bits and local"] = rank_qubits[::-1] + [q for q in range(n) if q not in rank_qubits][:3]
        for what, qubits in cases.items():
            got = sv.marginal(qubits)
            want = eng.marginal_probabilities([plan], [values], qubits)[0]
            assert np.max(np.abs(got - want)) <= 1e-14, f"{shards} shards, {buffers} buffers, {what}"
            assert np.array_equal(sv.marginal(qubits).view(np.uint64), got.view(np.uint64))
    finally:
        sv.close()


def test_sampler_marginals_and_the_sharded_route():
    from queasars_b200.primitives import B200SamplerV2, get_engine
    from queasars_b200.sharded import LocalShardedStatevector

    n = 14
    cases = [evqe_case(n, 3, 900 + i) for i in range(4)]
    circs, vals = [c for _, _, c in cases], [v for _, v, _ in cases]
    qubits = [5, 13, 0]
    smp = B200SamplerV2(coalesce=True)
    got = smp.marginal_probabilities(circs, vals, qubits)
    eng = get_engine(0)
    for row, c, v in zip(got, circs, vals):
        amps = eng.statevector(eng.compile(gl.from_circuit(c)), v)
        assert np.max(np.abs(row - np_marginal(np.abs(amps) ** 2, n, qubits))) <= 1e-13
    sharded = B200SamplerV2(devices=[0], shard_min_qubits=n, coalesce=False)
    sharded._sharded_state = lambda width, sv=LocalShardedStatevector(n, [eng] * 2, min_local=8): sv
    s_got = sharded.marginal_probabilities(circs, vals, qubits)
    assert np.max(np.abs(s_got - got)) <= 1e-14


def register_projection(k, qubits):
    out = np.zeros_like(k)
    for j, q in enumerate(qubits):
        if q is not None:
            out |= ((k >> q) & 1) << j
    return out


@pytest.mark.parametrize("kind", ["subset", "permuted", "two registers"])
def test_run_registers_at_20_qubits(kind):
    from queasars_b200.primitives import B200SamplerV2

    n, shots = 20, 10_000
    _, values, base = evqe_case(n, 3, 2000)
    if kind == "subset":
        circ = QuantumCircuit(n, 4).compose(base)
        circ.measure([2, 7, 11, 19], range(4))
        regs = [("c", [2, 7, 11, 19])]
    elif kind == "permuted":
        circ = QuantumCircuit(n, 5).compose(base)
        circ.measure([19, 0, 10, 3, 12], [3, 0, 4, 1, 2])
        regs = [("c", [0, 3, 12, 19, 10])]
    else:
        circ = QuantumCircuit(n, ClassicalRegister(3, "c"), ClassicalRegister(2, "job")).compose(base)
        circ.measure([1, 4, 9], [0, 1, 2])
        circ.measure([18, 6], [3, 4])
        regs = [("c", [1, 4, 9]), ("job", [18, 6])]
    res = B200SamplerV2(seed=21).run([(circ, values)], shots=shots).result()[0]
    full = B200SamplerV2(seed=21).sample_indices([base], [values], shots)[0]
    exact = B200SamplerV2()
    assert list(res.data.keys()) == [name for name, _ in regs]
    for name, qubits in regs:
        reg = res.data[name]
        assert reg.num_bits == len(qubits) and np.array_equal(reg.indices, register_projection(full, qubits))
        p = exact.marginal_probabilities([base], [values], qubits)[0]
        counts = np.bincount(reg.indices, minlength=p.size) / shots
        tv = 0.5 * np.abs(counts - p).sum()
        # E[TV] <= sqrt(2^m / shots) / 2 (Cauchy-Schwarz); the deviation above it is below 0.04 with probability 1 - 1e-13 (McDiarmid)
        assert tv <= 0.5 * math.sqrt(p.size / shots) + 0.04, f"{kind} {name}: TV {tv}"
    joined = res.join_data()
    assert joined.num_bits == sum(len(q) for _, q in regs)
