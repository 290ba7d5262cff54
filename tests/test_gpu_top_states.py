"""Most probable basis states on the device (``qb_top_states`` / ``Engine.top_states``, the sharded select of
``LocalShardedStatevector.top_states``, ``B200SamplerV2.top_states`` and ``measure_quasi_distributions(shots=None)``) against
the oracle: ``np.lexsort((k, -p))`` over the entries with p > 0 and p >= min_probability, p = re * re + im * im of the same
amplitudes read back with ``Engine.statevector`` / ``gather_logical`` -- bit for bit, since the device rounds p without FMA
contraction.  Wide sizes are also checked against the independent C oracle within the dtype's tolerance."""
import math
import threading

import numpy as np
import pytest

from oracle import c_oracle
from oracle import evqe_genome as og
from queasars_b200 import QuantumCircuit
from queasars_b200 import gate_list as gl
from tests.test_frontend_planner import build_circuit
from tests.test_gpu_wide_states import fit_or_skip
from tests.test_top_states_host import oracle_top

pytestmark = pytest.mark.gpu

GiB = 1 << 30
PASSES: dict = {}


@pytest.fixture(scope="module", autouse=True)
def report_passes():
    yield
    print("\ntop states: select passes per case", PASSES)


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
    return instr, list(values), gl.from_circuit(build_circuit(instr, n))


def assert_equal_top(got, want, what):
    assert np.array_equal(got[0], want[0]), f"{what}: indices {got[0][:8]} vs {want[0][:8]}"
    assert np.array_equal(got[1].view(np.uint64), want[1].view(np.uint64)), f"{what}: probabilities differ"


def assert_close_top(got, amps, m, what, rtol=1e-12):
    """For states of the same circuit computed in another batch composition (the sweeps may round differently): the entries
    agree with the oracle's within ``rtol``, and every index taken is at least as probable as the oracle's cut (knife edge)."""
    want = oracle_top(amps, m)
    p = amps.real * amps.real + amps.imag * amps.imag
    assert got[0].size == want[0].size, what
    assert np.allclose(got[1], p[got[0]], rtol=rtol, atol=0) and np.allclose(got[1], want[1], rtol=rtol, atol=0), what
    assert np.all(p[got[0]] >= want[1][-1] * (1 - rtol)) and np.all(np.diff(got[1]) <= 0), what


def limits_of(p, n):
    desc = np.sort(p[p > 0])[::-1]
    return [(m, mp) for m in (1, 7, 1024, min((1 << n) + 5, 1 << 20)) for mp in (0.0, float(desc[min(9, desc.size - 1)]), 1e-3)]


@pytest.mark.parametrize("dtype", ["complex128", "complex64"])
@pytest.mark.parametrize("n", [10, 16, 20, 24])
def test_random_individuals_against_the_oracle(engines, dtype, n):
    eng = engines[dtype]
    instr, values, gates = evqe_case(n, 4, 100 + n)
    plan = eng.compile(gates)
    amps = eng.statevector(plan, values)
    p = amps.real * amps.real + amps.imag * amps.imag
    if n >= 20:  # the device state itself against the C oracle
        _, ref = c_oracle.evaluate(instr, n, values, None, np.empty(1 << n, dtype=np.complex128))
        pref = ref.real**2 + ref.imag**2
        assert np.max(np.abs(p - pref)) <= (1e-12 if dtype == "complex128" else 1e-5) * max(1e-300, pref.max())
    for m, mp in limits_of(p, n):
        got = eng.top_states([plan], [values], m, mp)[0]
        assert_equal_top(got, oracle_top(amps, m, mp), f"{dtype} n={n} max_states={m} min_p={mp}")


def test_batch_of_32_repeated_and_recomposed(engines):
    eng = engines["complex128"]
    n = 20
    cases = [evqe_case(n, 3, 500 + i) for i in range(32)]
    plans = [eng.compile(g) for _, _, g in cases]
    vals = [v for _, v, _ in cases]
    for m in (1, 1024):
        whole = eng.top_states(plans, vals, m, 0.0)
        again = eng.top_states(plans, vals, m, 0.0)
        rev = eng.top_states(plans[::-1], vals[::-1], m, 0.0)[::-1]
        for i, (plan, v) in enumerate(zip(plans, vals)):
            assert_equal_top(again[i], whole[i], f"entry {i} max_states={m}, repeated call")
            amps = eng.statevector(plan, v)  # (a batch of one: its sweeps may round differently from the batch of 32)
            for got in (whole[i], rev[i], eng.top_states([plan], [v], m, 0.0)[0]):
                assert_close_top(got, amps, m, f"entry {i} max_states={m}")
            assert_equal_top(eng.top_states([plan], [v], m, 0.0)[0], oracle_top(amps, m), f"entry {i} max_states={m}, alone")


def dyadic(n, kind):
    circ = QuantumCircuit(n)
    if kind == "uniform":
        for q in range(n):
            circ.h(q)
    elif kind == "ghz":
        circ.h(0)
        for q in range(1, n):
            circ.cx(0, q)
    else:  # mixed: |+> on the even qubits, |1> on every third odd one, a rotation on qubit 1
        for q in range(0, n, 2):
            circ.h(q)
        for q in range(3, n, 6):
            circ.x(q)
        circ.ry(1.1, 1)
    return circ


@pytest.mark.parametrize("dtype", ["complex128", "complex64"])
@pytest.mark.parametrize("kind", ["uniform", "ghz", "mixed"])
def test_dyadic_states_with_exact_ties(engines, dtype, kind):
    eng = engines[dtype]
    n = 14
    plan = eng.compile(gl.from_circuit(dyadic(n, kind)))
    amps = eng.statevector(plan, [])
    p = amps.real * amps.real + amps.imag * amps.imag
    cut_in_ties = 0
    for m in (1, 2, 3, 7, 100, 1 << (n - 1), (1 << n) + 5):
        got = eng.top_states([plan], [[]], m, 0.0)[0]
        assert_equal_top(got, oracle_top(amps, m), f"{dtype} {kind} max_states={m}")
        cut_in_ties += 0 < got[1].size == m and np.count_nonzero(p == got[1][-1]) > np.count_nonzero(got[1] == got[1][-1])
    if kind == "uniform":
        got = eng.top_states([plan], [[]], 7, 0.0)[0]
        assert list(got[0]) == list(range(7))  # one run of 2^14 ties: the lowest indices
    if kind == "ghz":
        # (the X gates leave amplitudes of order 1e-17 elsewhere: a threshold keeps the two GHZ entries)
        assert list(eng.top_states([plan], [[]], 5, 1e-20)[0][0]) == [0, (1 << n) - 1]
    if kind != "ghz":
        assert cut_in_ties
    # min_probability equal to a tie run's p keeps the whole run
    mp = float(np.max(p))
    got = eng.top_states([plan], [[]], 1 << 20, mp)[0]
    assert_equal_top(got, oracle_top(amps, 1 << 20, mp), f"{dtype} {kind} min_p = max p")


def test_index_width_64_is_bit_identical():
    from queasars_b200.engine import Engine

    n = 20
    _, values, gates = evqe_case(n, 3, 77)
    narrow, wide = Engine(device=0), Engine(device=0)
    try:
        wide.set_index_width(64)
        a, b = narrow.compile(gates), wide.compile(gates)
        for m in (1, 1024):
            assert_equal_top(wide.top_states([b], [values], m)[0], narrow.top_states([a], [values], m)[0], f"64-bit index max_states={m}")
    finally:
        narrow.close(), wide.close()


def test_32_qubits_closed_form_on_64_bit_indices():
    """2^32 complex64 amplitudes: RY on qubits 0, 5 and 31, H on qubit 20, |0> elsewhere -- 16 entries with known p, a tie pair
    per pattern of the three rotated qubits, indices up to 2^32 - 1."""
    from queasars_b200.engine import Engine

    n = 32
    fit_or_skip((8 << n) + 2 * GiB, "a 32-qubit complex64 state")
    circ = QuantumCircuit(n)
    thetas = {0: 0.6, 5: 1.0, 31: 2.2}
    for q, t in thetas.items():
        circ.ry(t, q)
    circ.h(20)
    eng = Engine(device=0, dtype="complex64")
    try:
        plan = eng.compile(gl.from_circuit(circ))
        entries = []
        for bits in range(8):
            k, p = 0, 1.0
            for j, (q, t) in enumerate(thetas.items()):
                one = (bits >> j) & 1
                k |= one << q
                p *= math.sin(t / 2) ** 2 if one else math.cos(t / 2) ** 2
            entries += [(-p / 2, k), (-p / 2, k | (1 << 20))]
        entries.sort()
        for m in (1, 5, 16, 1024):
            idx, probs = eng.top_states([plan], [[]], m, 0.0)[0]
            want = entries[:m]
            # tie pairs come out in ascending index; the product of rounded factors may split a pair by an ulp only
            assert sorted(idx.tolist()) == sorted(k for _, k in want) and idx.size == len(want)
            assert np.allclose(probs, [-v for v, _ in want], rtol=2e-6, atol=0)
            assert np.all(np.diff(probs) <= 0)
            assert int(idx.max()) >= 1 << 31
    finally:
        eng.close()


@pytest.mark.parametrize("shards", [1, 2, 4, 8])
def test_local_sharded_state_after_swaps(shards):
    from queasars_b200.primitives import get_engine
    from queasars_b200.sharded import LocalShardedStatevector

    n = 16
    _, values, gates = evqe_case(n, 4, 900 + shards)
    sv = LocalShardedStatevector(n, [get_engine(0)] * shards, min_local=8)
    try:
        sv.run(gates, values)
        if shards > 1:
            assert sv.swaps_done and sv.position != list(range(n))
        full = sv.gather_logical()
        p = full.real * full.real + full.imag * full.imag
        for m, mp in limits_of(p, n):
            got = sv.top_states(m, mp)
            assert_equal_top(got, oracle_top(full, m, mp), f"{shards} shards max_states={m} min_p={mp}")
        PASSES[("sharded", shards)] = sv.top_passes
        # a sharded near-uniform superposition (the sweeps round the 2^16 equal magnitudes into a few runs of ties)
        circ = QuantumCircuit(n)
        for q in range(n - 1, -1, -1):
            circ.h(q)
        sv.reset()
        sv.run(gl.from_circuit(circ), [])
        full = sv.gather_logical()
        for m in (1, 7, 1000):
            assert_equal_top(sv.top_states(m), oracle_top(full, m), f"{shards} shards, H on every qubit, max_states={m}")
    finally:
        sv.close()


def test_sampler_routes_threads_device_sets_and_sharding():
    from queasars_b200 import _native
    from queasars_b200.evaluators import measure_quasi_distributions
    from queasars_b200.primitives import B200SamplerV2

    n = 14
    cases = [evqe_case(n, 3, 1200 + i) for i in range(6)]
    circs = [build_circuit(instr, n) for instr, _, _ in cases]
    vals = [v for _, v, _ in cases]
    smp = B200SamplerV2(devices="all")
    ref = B200SamplerV2(coalesce=False)
    want = ref.top_states(circs, vals, 16, 0.0)
    got = [None] * len(circs)

    def work(i):
        got[i] = smp.top_states([circs[i]], [vals[i]], 16, 0.0)[0]

    threads = [threading.Thread(target=work, args=(i,)) for i in range(len(circs))]
    [t.start() for t in threads]
    [t.join() for t in threads]
    for i in range(len(circs)):
        assert_equal_top(got[i], want[i], f"coalesced thread {i}")
    dists = measure_quasi_distributions(circs, vals, smp, None, max_states=16)
    for d, (idx, probs) in zip(dists, want):
        assert d.shots is None and list(d.keys()) == idx.tolist() and list(d.values()) == probs.tolist()
    # the sharded route (every device of the set, or two shards of one GPU): the same entries up to the rounding of the
    # unsharded plan's deferred phases
    sharded = B200SamplerV2(devices="all" if _native.device_count() > 1 else [0], shard_min_qubits=n, coalesce=False)
    if _native.device_count() == 1:
        from queasars_b200.primitives import get_engine
        from queasars_b200.sharded import LocalShardedStatevector

        sharded._sharded_state = lambda width, sv=LocalShardedStatevector(n, [get_engine(0)] * 2, min_local=8): sv
    for (idx, probs), (s_idx, s_probs) in zip(want, sharded.top_states(circs, vals, 16, 0.0)):
        assert np.array_equal(idx, s_idx) and np.allclose(probs, s_probs, rtol=1e-12, atol=0)


def test_35_qubits_on_8_gpus_closed_form():
    """Product state RY(theta) on every qubit: the C(n, j) states with j ones have p = s^j (1 - s)^(n - j), s = sin^2(theta / 2) <
    1/2, so the top states are 0, then the n states with one 1 in ascending index, then those with two."""
    from queasars_b200 import _native
    from queasars_b200.primitives import get_engine
    from queasars_b200.sharded import LocalShardedStatevector

    if _native.device_count() < 8:
        pytest.skip("35 qubits need 8 GPUs")
    n, theta = 35, 1.1
    circ = QuantumCircuit(n)
    for q in range(n):
        circ.ry(theta, q)
    sv = LocalShardedStatevector(n, [get_engine(d) for d in range(8)])
    try:
        sv.run(gl.from_circuit(circ), [])
        idx, probs = sv.top_states(1 + n)
        s = math.sin(theta / 2) ** 2
        # (the n one-hot states tie up to the rounding of their products: compared as a set)
        assert idx[0] == 0 and sorted(idx[1:].tolist()) == [1 << q for q in range(n)]
        assert np.allclose(probs, [(1 - s) ** n] + [s * (1 - s) ** (n - 1)] * n, rtol=1e-12, atol=0) and np.all(np.diff(probs) <= 0)
    finally:
        sv.close()
