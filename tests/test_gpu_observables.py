"""Several observables per state on the device (``qb_evaluate_observables``, ``Engine.expectation_many``,
``B200EstimatorV2.expectation_values_many`` and ``run()`` with an observables array) against the NumPy / C oracle and against
the single-observable route; determinism across runs, batch compositions, workspace limits and term chunking; the sharded
route; shaped sampler pubs; errors as the C-ABI returns them."""
import numpy as np
import pytest

from oracle import c_oracle
from oracle import evqe_genome as og
from oracle import qiskit_semantics as oq
from queasars_b200 import _native
from queasars_b200 import expectation as ex
from queasars_b200 import gate_list as gl
from queasars_b200.operators import SparsePauliOp
from tests.test_frontend_planner import build_circuit
from tests.test_gpu_parity import random_ising, tfim

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    from queasars_b200.engine import Engine

    return Engine(device=0, dtype="complex128")


def evqe_case(n, layers, seed):
    genome, values = og.random_individual(n, layers, True, seed)
    instr = og.individual_circuit(genome, values)
    return instr, list(values), build_circuit(instr, n)


def state_of(instr, n, values):
    if n < 16:
        return oq.statevector(instr, n, values)
    _, state = c_oracle.evaluate(instr, n, values, None, np.empty(1 << n, dtype=np.complex128))
    return state


def reference(state, n, terms):
    return oq.estimator_expectation(state, terms) if n < 16 else c_oracle.pauli_sum(state, n, terms)


def label(n, paulis: dict) -> str:
    lab = ["I"] * n
    for q, p in paulis.items():
        lab[n - 1 - q] = p
    return "".join(lab)


def random_strings(n, k, seed, width=None):
    """k operators of 1-3 random X / Y / Z strings (Y phases included); ``width``: qubits touched per string."""
    rng = np.random.default_rng(seed)
    ops = []
    for _ in range(k):
        terms = []
        for _ in range(int(rng.integers(1, 4))):
            qs = rng.choice(n, size=width or int(rng.integers(1, n + 1)), replace=False)
            terms.append((label(n, {int(q): str(rng.choice(list("XYZ"))) for q in qs}), float(rng.normal())))
        ops.append(terms)
    return ops


def correlators(n):
    """All <Z_i> and <Z_i Z_j>."""
    ops = [[(label(n, {i: "Z"}), 1.0)] for i in range(n)]
    ops += [[(label(n, {i: "Z", j: "Z"}), 1.0)] for i in range(n) for j in range(i + 1, n)]
    return ops


def tfim_parts(n):
    return [tfim(n)] + [[(label(n, {i: "X"}), 1.0)] for i in range(n)] + [[(label(n, {i: "Z"}), 1.0)] for i in range(n)]


def jssp_parts(entry):
    """The JSSP energy and its diagonal terms split three ways (stand-ins for the encoding / overlap / precedence penalties)."""
    z, c = ex.merge_diagonal_terms(np.asarray(entry["z_masks"], dtype=np.uint64), np.asarray(entry["coeffs"], dtype=np.float64))
    n = int(entry["n_qubits"])
    terms = [(oq_label(n, int(zz)), float(cc)) for zz, cc in zip(z, c)]
    return [terms] + [terms[k::3] for k in range(3)]


def oq_label(n, zmask):
    return "".join("Z" if (zmask >> q) & 1 else "I" for q in range(n - 1, -1, -1))


def spo(terms):
    return SparsePauliOp.from_list(terms)


def assert_close(got, want, rtol):
    err = abs(got - want) / max(1.0, abs(want))
    assert err <= rtol, f"got {got!r}, want {want!r} (rel {err:.2e})"


# ------------------------------------------------------------------------------------ parity
@pytest.mark.parametrize("n", [4, 8, 12, 16, 20])
def test_random_individuals_against_the_oracle(engine, n):
    obs = random_strings(n, 12, 100 + n) + [tfim(n), random_ising(n)] + tfim_parts(n)[1:4]
    if n <= 12:
        obs += correlators(n)
    handle = engine.observables([spo(t) for t in obs])
    cases = [evqe_case(n, 2 + s % 4, 3000 + 17 * n + s) for s in range(6)]
    plans = [engine.compile(gl.from_circuit(c)) for _, _, c in cases]
    got = engine.expectation_many(plans, [v for _, v, _ in cases], handle)
    assert got.shape == (len(cases), len(obs))
    for row, (instr, values, _) in zip(got, cases):
        state = state_of(instr, n, values)
        for g, terms in zip(row, obs):
            assert_close(g, reference(state, n, terms), 1e-10)


@pytest.mark.parametrize("n,which", [(20, "correlators"), (22, "random"), (24, "tfim")])
def test_wide_states_against_the_c_oracle(engine, n, which):
    obs = {"correlators": correlators, "random": lambda n: random_strings(n, 16, 7 * n), "tfim": tfim_parts}[which](n)
    handle = engine.observables([spo(t) for t in obs])
    instr, values, circ = evqe_case(n, 3, 4000 + n)
    got = engine.expectation_many([engine.compile(gl.from_circuit(circ))], [values], handle)[0]
    state = state_of(instr, n, values)
    for g, terms in zip(got, obs):
        assert_close(g, c_oracle.pauli_sum(state, n, terms), 1e-10)


def test_jssp_26q_parts(engine, jssp_golden):
    obs = jssp_parts(jssp_golden["jssp_26q"])
    n = 26
    handle = engine.observables([spo(t) for t in obs])
    assert handle.diagonal
    instr, values, circ = evqe_case(n, 3, 26)
    got = engine.expectation_many([engine.compile(gl.from_circuit(circ), drop_final_phases=True)], [values], handle)[0]
    state = state_of(instr, n, values)
    for g, terms in zip(got, obs):
        assert_close(g, c_oracle.pauli_sum(state, n, terms), 1e-10)
    assert_close(got[0], sum(got[1:]), 1e-12)


def test_complex64(engine):
    from queasars_b200.engine import Engine

    e64 = Engine(device=0, dtype="complex64")
    n = 14
    obs = random_strings(n, 8, 5) + tfim_parts(n)
    handle = e64.observables([spo(t) for t in obs])
    cases = [evqe_case(n, 3, 600 + s) for s in range(4)]
    got = e64.expectation_many([e64.compile(gl.from_circuit(c)) for _, _, c in cases], [v for _, v, _ in cases], handle)
    for row, (instr, values, _) in zip(got, cases):
        state = state_of(instr, n, values)
        for g, terms in zip(row, obs):
            assert_close(g, reference(state, n, terms), 1e-4)


# ------------------------------------------------------------------------------------ agreement with the single-observable route
@pytest.mark.parametrize("n", [6, 13, 20])
def test_matches_the_single_observable_route(engine, n):
    obs = random_strings(n, 10, 40 + n) + random_strings(n, 4, 41 + n, width=n) + tfim_parts(n)[:6] + [random_ising(n)]
    ops = [spo(t) for t in obs]
    handle = engine.observables(ops)
    cases = [evqe_case(n, 2 + s % 3, 5000 + n + s) for s in range(5)]
    plans = [engine.compile(gl.from_circuit(c)) for _, _, c in cases]
    params = [v for _, v, _ in cases]
    got = engine.expectation_many(plans, params, handle)
    for j, op in enumerate(ops):
        want = engine.expectation(plans, params, engine.hamiltonian(op))
        for i in range(len(cases)):
            assert_close(got[i, j], want[i], 1e-12)


# ------------------------------------------------------------------------------------ planner coverage and determinism
def big_diagonal(n, count, seed):
    rng = np.random.default_rng(seed)
    zs = rng.choice(np.arange(1, 1 << n), size=count, replace=False)
    return SparsePauliOp._raw(n, [0] * count, [int(z) for z in zs], rng.normal(size=count).tolist())


def test_planner_coverage_chunking_and_determinism(engine):
    from queasars_b200.engine import Engine

    # 16 q: a row alone and in a batch of 32 get the same sweep launch shape, hence bit-identical states (at 20 q the tiles per
    # sweep CTA follow the batch size and the states themselves may differ in the last bit, on the single-observable route too)
    n = 16
    wide = [[(label(n, {q: "X" for q in range(n)}), 0.5), (label(n, {0: "Y", 15: "Y", 7: "Z"}), 1.5)]]  # wider than a tile
    inside = tfim_parts(n)[1:5]  # single-qubit X: inside a tile
    big = big_diagonal(n, 2100, 9)  # one group of more than 2 000 strings
    ops = [spo(t) for t in wide + inside] + [big, spo(random_ising(n))]
    handle = engine.observables(ops)
    assert handle.n_terms > 2100
    cases = [evqe_case(n, 2 + s % 4, 7000 + s) for s in range(32)]
    plans = [engine.compile(gl.from_circuit(c)) for _, _, c in cases]
    params = [v for _, v, _ in cases]
    batch = engine.expectation_many(plans, params, handle)
    again = engine.expectation_many(plans, params, handle)
    assert np.array_equal(batch, again)  # across runs
    for i in (0, 13, 31):  # a row alone vs the same row in the batch of 32
        alone = engine.expectation_many([plans[i]], [params[i]], handle)[0]
        assert np.array_equal(alone, batch[i])
    # a workspace of six 1 MiB states: the batch is split into pieces of five, and the partials scratch left next to them holds
    # a few hundred strings, so every tile sweep and wide group is evaluated in several launches over string ranges
    small = Engine(device=0, dtype="complex128", workspace_limit=6 << 20)
    split = small.expectation_many([small.compile(gl.from_circuit(c)) for _, _, c in cases], params, small.observables(ops))
    assert np.array_equal(split, batch)
    instr, values, _ = cases[5]
    state = state_of(instr, n, values)
    for g, op in zip(batch[5], ops):
        assert_close(g, c_oracle.pauli_sum(state, n, op.to_list()), 1e-10)


def test_term_chunking_at_20_qubits(engine):
    """At 20 q x 32 states the 2 100-string group exceeds the 256 MiB partials scratch of one launch; the same batch evaluated in
    pieces of two states is not chunked.  Both equal the oracle, and each piece equals the chunked batch where its rows do."""
    n = 20
    ops = [big_diagonal(n, 2100, 11), spo(tfim(n))]
    handle = engine.observables(ops)
    cases = [evqe_case(n, 2 + s % 4, 7100 + s) for s in range(32)]
    plans = [engine.compile(gl.from_circuit(c)) for _, _, c in cases]
    params = [v for _, v, _ in cases]
    batch = engine.expectation_many(plans, params, handle)
    for i in (0, 17):
        state = state_of(cases[i][0], n, cases[i][1])
        for g, op in zip(batch[i], ops):
            assert_close(g, c_oracle.pauli_sum(state, n, op.to_list()), 1e-10)
    pair = engine.expectation_many(plans[:2], params[:2], handle)
    for j, op in enumerate(ops):
        want = engine.expectation(plans[:2], params[:2], engine.hamiltonian(op))
        for i in range(2):
            assert_close(pair[i, j], want[i], 1e-12)
            assert_close(batch[i, j], want[i], 1e-12)


def test_device_sets_and_primitive_route(engine):
    from queasars_b200 import B200EstimatorV2

    n = 12
    ops = [spo(t) for t in random_strings(n, 6, 77) + tfim_parts(n)[:3]]
    cases = [evqe_case(n, 2 + s % 3, 8000 + s) for s in range(12)]
    circuits, params = [c for _, _, c in cases], [v for _, v, _ in cases]
    one = B200EstimatorV2(coalesce=False).expectation_values_many(circuits, params, ops)
    every = B200EstimatorV2(devices="all").expectation_values_many(circuits, params, ops)
    assert np.array_equal(one, every)
    plans = [engine.compile(gl.from_circuit(c)) for c in circuits]  # (no cached prefix state: rounding may differ in the last bits)
    direct = engine.expectation_many(plans, params, engine.observables(ops))
    assert np.allclose(one, direct, rtol=1e-12, atol=1e-12)


def test_sharded_route():
    from queasars_b200 import B200EstimatorV2

    n = 14
    obs = random_strings(n, 5, 90) + tfim_parts(n)[:3]
    ops = [spo(t) for t in obs]
    cases = [evqe_case(n, 3, 9000 + s) for s in range(2)]
    est = B200EstimatorV2(devices="all", coalesce=False, shard_min_qubits=n)
    got = est.expectation_values_many([c for _, _, c in cases], [v for _, v, _ in cases], ops)
    for row, (instr, values, _) in zip(got, cases):
        state = state_of(instr, n, values)
        for g, terms in zip(row, obs):
            assert_close(g, reference(state, n, terms), 1e-10)


# ------------------------------------------------------------------------------------ primitives
def test_run_broadcasting_noise_and_stds():
    from queasars_b200 import B200EstimatorV2

    n = 10
    instr, values, circ = evqe_case(n, 3, 321)
    obs = [[label(n, {0: "Z"})], [label(n, {3: "X", 4: "Y"})], [{label(n, {1: "Z", 2: "Z"}): 0.5}]]
    rng = np.random.default_rng(2)
    pvals = np.stack([np.asarray(values) + rng.normal(scale=0.1, size=len(values)) for _ in range(4)])
    exact = B200EstimatorV2().run([(circ, obs, pvals)]).result()[0]
    assert exact.data.evs.shape == (3, 4) and exact.data.stds.shape == (3, 4) and np.all(exact.data.stds == 0.0)
    for r in range(4):
        state = oq.statevector(instr, n, pvals[r])
        for o, terms in enumerate([[(obs[0][0], 1.0)], [(obs[1][0], 1.0)], [(label(n, {1: "Z", 2: "Z"}), 0.5)]]):
            assert_close(exact.data.evs[o, r], oq.estimator_expectation(state, terms), 1e-10)
    noisy = B200EstimatorV2(seed=4).run([(circ, obs, pvals)], precision=0.05).result()[0]
    assert np.array_equal(noisy.data.evs, np.random.default_rng(4).normal(exact.data.evs, 0.05))
    assert np.all(noisy.data.stds == 0.05) and noisy.data.stds.shape == (3, 4)


def test_shaped_sampler_pub():
    from queasars_b200 import B200SamplerV2

    n = 9
    instr, values, circ = evqe_case(n, 3, 55)
    circ.measure_all()
    rng = np.random.default_rng(8)
    pvals = np.asarray(values) + rng.normal(scale=0.2, size=(2, 3, len(values)))
    meas = B200SamplerV2(seed=13).run([(circ, pvals)], shots=500).result()[0].data.meas
    assert meas.shape == (2, 3) and meas.num_shots == 500
    uniforms = np.random.default_rng(13).random(500)
    for pos in np.ndindex(2, 3):
        want = oq.sample_indices(oq.statevector(instr, n, pvals[pos]), 500, uniforms=uniforms)
        assert np.sum(meas.indices[pos] != want) <= 1  # ("<= 1 boundary flip": device and NumPy cumulative sums differ in the last bits)
    assert sum(meas.get_counts().values()) == 3000


# ------------------------------------------------------------------------------------ errors
def test_errors(engine):
    import ctypes

    from queasars_b200.engine import Engine

    n = 8
    handle = engine.observables([spo(tfim(n)), spo(random_ising(n))])
    _, values, circ = evqe_case(n + 1, 2, 1)
    with pytest.raises(_native.QbError) as err:
        engine.expectation_many([engine.compile(gl.from_circuit(circ))], [values], handle)
    assert err.value.code == _native.QB_ERR_INVALID
    lib, out = engine._lib, ctypes.c_int64()
    offs = np.zeros(1, dtype=np.int64)
    assert lib.qb_observables_create(engine._ctx, n, 0, _native.ptr(offs), None, None, None, None, ctypes.byref(out)) == _native.QB_ERR_INVALID
    bad = np.array([0, 2, 1], dtype=np.int64)
    x = np.zeros(2, dtype=np.uint64)
    c = np.ones(2)
    assert lib.qb_observables_create(engine._ctx, n, 2, _native.ptr(bad), _native.ptr(x), _native.ptr(x), _native.ptr(c), None, ctypes.byref(out)) == _native.QB_ERR_INVALID
    far = np.array([0, 1 << n], dtype=np.uint64)
    two = np.array([0, 2], dtype=np.int64)
    assert lib.qb_observables_create(engine._ctx, n, 1, _native.ptr(two), _native.ptr(far), _native.ptr(x), _native.ptr(c), None, ctypes.byref(out)) == _native.QB_ERR_INVALID
    res = np.zeros(4)
    ids = np.array([123456789], dtype=np.int64)
    assert lib.qb_evaluate_observables(engine._ctx, 1, _native.ptr(ids), _native.ptr(res), _native.ptr(offs), handle.obs_id, _native.ptr(res)) == _native.QB_ERR_NOT_FOUND
    assert lib.qb_observables_destroy(engine._ctx, 987654321) == _native.QB_ERR_NOT_FOUND
    tiny = Engine(device=0, dtype="complex128", workspace_limit=1 << 20)  # smaller than one 17-qubit state
    _, values, circ = evqe_case(17, 2, 2)
    with pytest.raises(_native.QbError) as err:
        tiny.expectation_many([tiny.compile(gl.from_circuit(circ))], [values], tiny.observables([spo(tfim(17))]))
    assert err.value.code == _native.QB_ERR_MEMORY and "bytes" in str(err.value)
