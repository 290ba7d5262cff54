"""Host logic of several observables per estimator pub on CPU: coercion of the observable forms, V2 broadcasting, the union /
CSR combination of ``qb_observables_create``, the coalescing key, the device split, the single-observable route, and shaped
sampler pubs -- with a ``FakeEngine`` whose ``observables`` / ``expectation_many`` evaluate every string with the oracle."""
import threading

import numpy as np
import pytest

from oracle import evqe_genome as og
from oracle import qiskit_semantics as oq
from queasars_b200 import containers as ct
from queasars_b200 import primitives as pr
from queasars_b200.engine import ObservablesHandle, observable_terms, observable_union
from queasars_b200.operators import SparsePauliOp
from tests.fake_engine import FakeEngine, _state
from tests.test_frontend_planner import build_circuit


class ManyFakeEngine(FakeEngine):
    def __init__(self, device=0, dtype="complex128"):
        super().__init__(device, dtype)
        self.calls = []
        self._sets = {}

    def expectation(self, plans, params, ham):
        self.calls.append(("expectation", len(plans)))
        return super().expectation(plans, params, ham)

    def observables(self, operators):
        n, x, z, c, offsets = observable_terms(operators)
        oid = self._new_id()
        self._sets[oid] = (n, observable_union(x, z, c, offsets))
        return ObservablesHandle(oid, n, len(offsets) - 1, not bool(np.any(x)), len(self._sets[oid][1][0]))

    def expectation_many(self, plans, params, handle):
        self.calls.append(("many", len(plans), handle.n_obs))
        n, (ux, uz, row_begin, cols, coeffs) = self._sets[handle.obs_id]
        out = np.empty((len(plans), handle.n_obs))
        for i, (plan, vals) in enumerate(zip(plans, params)):
            vals = np.asarray(vals, dtype=np.float64).reshape(-1)
            if vals.size != plan.n_params:
                raise ValueError(f"circuit has {plan.n_params} parameters but {vals.size} values were given")
            st = _state(self._plans[plan.plan_id], vals)
            idx = np.arange(st.size, dtype=np.uint64)
            pt = []
            for x, z in zip(ux, uz):
                sign = 1.0 - 2.0 * oq._parity(idx & np.uint64(z))
                ny = bin(int(x) & int(z)).count("1")
                pt.append(((1j**ny) * np.sum(np.conj(st[(idx ^ np.uint64(x)).astype(np.int64)]) * sign * st)).real)
            for j in range(handle.n_obs):
                out[i, j] = sum(coeffs[e] * pt[cols[e]] for e in range(row_begin[j], row_begin[j + 1]))
        return out


@pytest.fixture()
def fake_engines(monkeypatch):
    made = {}

    def get_engine(device=0, dtype="complex128"):
        return made.setdefault((device, dtype), ManyFakeEngine(device, dtype))

    monkeypatch.setattr(pr, "get_engine", get_engine)
    monkeypatch.setattr(pr._native, "device_count", lambda: 3)
    return made


def case(n, layers, seed):
    genome, values = og.random_individual(n, layers, True, seed)
    instr = og.individual_circuit(genome, values)
    return instr, list(values), build_circuit(instr, n)


def labels(n, seed, k):
    rng = np.random.default_rng(seed)
    return ["".join(rng.choice(list("IXYZ"), n)) for _ in range(k)]


def oracle_evs(instr, values, n, ops):
    st = oq.statevector(instr, n, values)
    return np.array([oq.estimator_expectation(st, op.to_list()) for op in ops])


def calls(engines, kind):
    return [c for e in engines.values() for c in e.calls if c[0] == kind]


def test_observable_forms_are_coerced():
    n = 3
    spo = SparsePauliOp.from_list([("XYZ", 0.5), ("III", -1.0)])
    ops, shape = pr._observables_array([spo, {"ZZI": 2.0, "XII": 1.0}, "YYX"])
    assert shape == (3,) and ops[0] is spo
    assert ops[1].to_list() == [("ZZI", 2.0), ("XII", 1.0)]
    assert ops[2].to_list() == [("YYX", 1.0)]
    ops, shape = pr._observables_array([["ZII", "IZI"], [{"IIZ": 1.0}, spo]])
    assert shape == (2, 2) and [o.num_qubits for o in ops] == [n] * 4

    class ObservablesArray:  # qiskit's: tolist() gives nested {label: coeff} dicts
        def __init__(self, items):
            self._items = items

        def tolist(self):
            return self._items

    ops, shape = pr._observables_array(ObservablesArray([[{"ZII": 1.0}], [{"XXI": 0.5, "IIY": 0.25}]]))
    assert shape == (2, 1) and ops[1].to_list() == [("XXI", 0.5), ("IIY", 0.25)]
    assert pr._observables_array("ZZZ")[1] == () and pr._observables_array(spo)[1] == ()
    with pytest.raises(ValueError):
        pr._observables_array([["ZII", "IZI"], ["IIZ"]])  # ragged
    with pytest.raises(TypeError):
        pr._observables_array([1.5, "ZZZ"])


def test_union_and_rows():
    a = SparsePauliOp.from_list([("XZ", 1.0), ("II", 0.5), ("XZ", 2.0), ("YY", -1.0)])  # duplicate within
    b = SparsePauliOp.from_list([("YY", 3.0), ("ZI", 1.5), ("II", 0.25)])  # duplicates across, identity again
    c = SparsePauliOp.from_list([("ZI", 1.0 + 2.0j)])  # only Re(c) counts
    n, x, z, coeffs, offsets = observable_terms([a, b, c])
    assert n == 2 and offsets.tolist() == [0, 3, 6, 7]  # (duplicates merged per operator)
    ux, uz, row_begin, cols, cf = observable_union(x, z, coeffs, offsets)
    strings = [(int(p), int(q)) for p, q in zip(ux, uz)]
    assert strings == [(0b10, 0b01), (0, 0), (0b11, 0b11), (0, 0b10)]  # XZ, II, YY, ZI: first appearance
    assert row_begin.tolist() == [0, 3, 6, 7]
    assert cols.tolist() == [0, 1, 2, 1, 2, 3, 3]  # ascending string order in every row
    assert cf.tolist() == [3.0, 0.5, -1.0, 0.25, 3.0, 1.5, 1.0]
    raw = observable_union(np.array([1, 1, 0], dtype=np.uint64), np.array([0, 0, 0], dtype=np.uint64), np.array([1.0, 2.0, 4.0]), [0, 3])
    assert raw[3].tolist() == [0, 1] and raw[4].tolist() == [3.0, 4.0]  # (the native side sums duplicates too)
    with pytest.raises(ValueError):
        observable_terms([a, SparsePauliOp.from_list([("ZZZ", 1.0)])])


@pytest.mark.parametrize("obs_shape,param_shape", [((4,), ()), ((4, 1), (3,)), ((4,), (4,)), ((2, 2), (2, 1))])
def test_broadcast_shapes(fake_engines, obs_shape, param_shape):
    n = 4
    est = pr.B200EstimatorV2()
    size = int(np.prod(obs_shape))
    labs = labels(n, 5, size)
    obs = np.array(labs, dtype=object).reshape(obs_shape).tolist()
    instr, _, circ = case(n, 2, 3)
    n_params = circ.num_parameters
    rng = np.random.default_rng(1)
    pvals = rng.uniform(-np.pi, np.pi, param_shape + (n_params,))
    res = est.run([(circ, obs, pvals)]).result()[0]
    shape = np.broadcast_shapes(obs_shape, param_shape)
    assert res.data.evs.shape == shape and res.data.stds.shape == shape and res.data.shape == shape
    ops = [SparsePauliOp(l) for l in labs]
    o_idx = np.broadcast_to(np.arange(size).reshape(obs_shape), shape)
    p_rows = pvals.reshape(-1, n_params)
    p_idx = np.broadcast_to(np.arange(len(p_rows)).reshape(param_shape), shape)
    for pos in np.ndindex(shape):
        want = oracle_evs(instr, p_rows[p_idx[pos]], n, [ops[o_idx[pos]]])[0]
        assert res.data.evs[pos] == pytest.approx(want, rel=1e-12, abs=1e-12)
    # every distinct parameter row simulated once, with every distinct observable
    many = calls(fake_engines, "many")
    assert sum(c[1] for c in many) == len(p_rows) and {c[2] for c in many} == {len(set(labs))}


def test_incompatible_shapes_and_widths(fake_engines):
    n = 4
    est = pr.B200EstimatorV2()
    _, values, circ = case(n, 2, 4)
    pvals = np.tile(values, (3, 1))
    with pytest.raises(ValueError):
        est.run([(circ, ["ZIII", "IZII"], pvals)]).result()
    with pytest.raises(ValueError):
        est.run([(circ, ["ZIII", "IZIII"], values)]).result()
    with pytest.raises(ValueError):
        est.expectation_values_many([circ], [values], [SparsePauliOp("ZZZ"), SparsePauliOp("XXX")])


def test_precision_noise_and_stds(fake_engines):
    n = 4
    est = pr.B200EstimatorV2(seed=11)
    instr, values, circ = case(n, 2, 6)
    labs = ["ZIII", "XXII", "IIYY"]
    res = est.run([(circ, labs, values)], precision=0.1).result()[0]
    exact = oracle_evs(instr, values, n, [SparsePauliOp(l) for l in labs])
    want = np.random.default_rng(11).normal(exact, 0.1)
    assert res.data.evs == pytest.approx(want, rel=1e-10)
    assert res.data.stds.shape == (3,) and np.all(res.data.stds == 0.1)


def test_single_observable_keeps_its_route(fake_engines):
    n = 4
    est = pr.B200EstimatorV2()
    instr, values, circ = case(n, 2, 7)
    op = SparsePauliOp.from_list([("ZZII", 1.0), ("XIIX", 0.5)])
    seen = []
    original = est.expectation_values

    def spy(circuits, params, operator):
        seen.append(operator)
        return original(circuits, params, operator)

    est.expectation_values = spy
    for obs in (op, [op], {"ZZII": 1.0, "XIIX": 0.5}):
        res = est.run([(circ, obs, values)]).result()[0]
        assert res.data.evs.shape == ()
        assert float(res.data.evs) == pytest.approx(oracle_evs(instr, values, n, [op])[0], rel=1e-12)
    assert len(seen) == 3 and not calls(fake_engines, "many")
    res = est.run([(circ, [op, op], values)]).result()[0]  # two elements: the set route, one distinct observable
    assert len(seen) == 3 and calls(fake_engines, "many")[-1][2] == 1
    assert res.data.evs.shape == (2,) and res.data.evs[0] == res.data.evs[1]


def test_coalescing_key(fake_engines):
    n = 4
    est = pr.B200EstimatorV2()
    set_a = [SparsePauliOp(l) for l in labels(n, 1, 3)]
    set_b = [SparsePauliOp(l) for l in labels(n, 2, 3)]
    keys = []
    original = est._execute

    def spy(key, payloads):
        keys.append((key, len(payloads)))
        return original(key, payloads)

    est._execute = spy
    est._queue
    est._queue_obj._execute = spy
    cases = [case(n, 2, 50 + s) for s in range(8)]
    sets = [set_a, set_b] * 4
    results = [None] * len(cases)
    gate = threading.Barrier(len(cases))

    def work(i):
        gate.wait()
        _, values, circ = cases[i]
        results[i] = est.expectation_values_many([circ], [values], sets[i])[0]

    threads = [threading.Thread(target=work, args=(i,)) for i in range(len(cases))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for (instr, values, _), ops, got in zip(cases, sets, results):
        assert got == pytest.approx(oracle_evs(instr, values, n, ops), rel=1e-12, abs=1e-12)
    ids = {tuple(id(o) for o in set_a), tuple(id(o) for o in set_b)}
    for key, _ in keys:
        assert key[0] == "many" and key[1] in ids  # payloads of one call always share a set
    assert sum(count for _, count in keys) == len(cases)
    assert est._execute(("many", keys[0][0][1], keys[0][0][2]), [(set_a, [cases[0][2]], [cases[0][1]])])[0].shape == (1, 3)
    # an in-place edit of a coefficient changes the key and rebuilds the device form
    before = est.observables_for(set_a)
    set_a[0]._c[0] = 2.0
    assert est.observables_for(set_a) is not before


def test_ordered_device_split(fake_engines):
    n = 4
    est = pr.B200EstimatorV2(devices="all")
    ops = [SparsePauliOp(l) for l in labels(n, 9, 5)]
    cases = [case(n, 1 + s % 3, 60 + s) for s in range(9)]
    got = est.expectation_values_many([c for _, _, c in cases], [v for _, v, _ in cases], ops)
    assert got.shape == (9, 5)
    for row, (instr, values, _) in zip(got, cases):
        assert row == pytest.approx(oracle_evs(instr, values, n, ops), rel=1e-12, abs=1e-12)
    assert sum(1 for e in fake_engines.values() if any(c[0] == "many" for c in e.calls)) > 1
    assert est.expectation_values_many([], [], ops).shape == (0, 5)


def test_sharded_route(fake_engines, monkeypatch):
    n = 4
    est = pr.B200EstimatorV2(shard_min_qubits=n)
    ops = [SparsePauliOp(l) for l in labels(n, 3, 4)]
    cases = [case(n, 2, 70 + s) for s in range(2)]

    class FakeSharded:
        def reset(self):
            pass

        def run(self, gates, params):
            self.st = _state(gates, params)

        def expectation(self, op):
            return oq.estimator_expectation(self.st, op.to_list())

    monkeypatch.setattr(est, "_sharded_state", lambda width: FakeSharded())
    got = est.expectation_values_many([c for _, _, c in cases], [v for _, v, _ in cases], ops)
    for row, (instr, values, _) in zip(got, cases):
        assert row == pytest.approx(oracle_evs(instr, values, n, ops), rel=1e-12, abs=1e-12)
    assert not calls(fake_engines, "many")


class _ShardedOracle:
    """Stand-in for ``LocalShardedStatevector``: the oracle's statevector of the last run."""

    def reset(self):
        self.st = None

    def run(self, gates, params):
        self.st = _state(gates, params)

    def expectation(self, op):
        return oq.estimator_expectation(self.st, op.to_list())

    def sample(self, shots, uniforms):
        return oq.sample_indices(self.st, shots, uniforms=uniforms)


def test_sharded_single_operator_route(fake_engines, monkeypatch):
    n = 4
    est = pr.B200EstimatorV2(shard_min_qubits=n)
    op = SparsePauliOp.from_list([(l, 0.5 + k) for k, l in enumerate(labels(n, 11, 4))])
    cases = [case(n, 2, 90 + s) for s in range(3)]
    monkeypatch.setattr(est, "_sharded_state", lambda width: _ShardedOracle())
    got = est.expectation_values([c for _, _, c in cases], [v for _, v, _ in cases], op)
    assert got.shape == (3,)
    for ev, (instr, values, _) in zip(got, cases):
        assert ev == pytest.approx(oracle_evs(instr, values, n, [op])[0], rel=1e-12, abs=1e-12)
    res = est.run([(cases[0][2], op, [cases[0][1], cases[0][1]])]).result()[0]
    assert res.data.evs.shape == (2,) and res.data.evs[1] == pytest.approx(got[0], rel=1e-12, abs=1e-12)
    assert not calls(fake_engines, "expectation") and not calls(fake_engines, "many")


def test_sharded_sampler_shots(fake_engines, monkeypatch):
    n, shots = 4, 96
    cases = [case(n, 2, 100 + s) for s in range(3)]
    circuits, values = [c for _, _, c in cases], [v for _, v, _ in cases]
    states = [oq.statevector(instr, n, v) for instr, v, _ in cases]
    # an int seed: a fresh generator per circuit, every row drawn from the same uniforms
    smp = pr.B200SamplerV2(seed=9, shard_min_qubits=n)
    monkeypatch.setattr(smp, "_sharded_state", lambda width: _ShardedOracle())
    got = smp.sample_indices(circuits, values, shots)
    uniforms = np.random.default_rng(9).random(shots)
    assert got.shape == (3, shots) and got.dtype == np.int64
    for row, st in zip(got, states):
        assert row.tolist() == oq.sample_indices(st, shots, uniforms=uniforms).tolist()
    # a Generator seed: consumed row after row in submission order
    smp = pr.B200SamplerV2(seed=np.random.default_rng(9), shard_min_qubits=n)
    monkeypatch.setattr(smp, "_sharded_state", lambda width: _ShardedOracle())
    got = smp.sample_indices(circuits, values, shots)
    gen = np.random.default_rng(9)
    for row, st in zip(got, states):
        assert row.tolist() == oq.sample_indices(st, shots, uniforms=gen.random(shots)).tolist()
    assert not any(e.calls for e in fake_engines.values())


@pytest.mark.parametrize("shape", [(3,), (2, 2)])
def test_shaped_sampler_pub(fake_engines, shape):
    n = 4
    instr, _, circ = case(n, 2, 80)
    circ.measure_all()
    rng = np.random.default_rng(3)
    pvals = rng.uniform(-np.pi, np.pi, shape + (circ.num_parameters,))
    res = pr.B200SamplerV2(seed=5).run([(circ, pvals)], shots=64).result()[0]
    meas = res.data.meas
    assert res.data.shape == shape and meas.shape == shape and meas.num_shots == 64 and meas.indices.shape == shape + (64,)
    uniforms = np.random.default_rng(5).random(64)  # an int seed: every bound circuit gets the same uniforms
    pooled = []
    for pos in np.ndindex(shape):
        st = oq.statevector(instr, n, pvals[pos])
        want = oq.sample_indices(st, 64, uniforms=uniforms)
        assert meas.indices[pos].tolist() == want.tolist()
        assert meas.get_int_counts(pos) == {int(v): int(c) for v, c in zip(*np.unique(want, return_counts=True))}
        pooled.extend(want.tolist())
    assert sum(meas.get_counts().values()) == 64 * int(np.prod(shape))
    assert meas.get_int_counts() == {int(v): int(c) for v, c in zip(*np.unique(pooled, return_counts=True))}
    assert len(meas.get_bitstrings()) == len(pooled) and len(meas.get_bitstrings(tuple(0 for _ in shape))) == 64


def test_zero_dimensional_register_unchanged():
    reg = ct.ShotRegister(np.array([3, 1, 3]), 2)
    assert reg.shape == () and reg.num_shots == 3 and reg.indices.shape == (3,)
    assert reg.get_counts() == {"11": 2, "01": 1} and reg.get_bitstrings() == ["11", "01", "11"]
