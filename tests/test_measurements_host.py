"""CPU tests of final measurements into classical registers: the circuit stand-in's registers and ``measure``, the measurement map
``gate_list.final_measurements``, the per-register read-out of ``B200SamplerV2.run`` (through the NumPy fake engine),
``join_data``, and the host side of ``marginal_probabilities`` (validation, routing, the sharded sum)."""
import numpy as np
import pytest

from oracle import evqe_genome as og
from oracle import qiskit_semantics as oq
from queasars_b200 import containers as ct
from queasars_b200 import gate_list as gl
from queasars_b200 import primitives as pr
from queasars_b200.circuit import ClassicalRegister, Clbit, Instruction, QuantumCircuit
from queasars_b200.sharded import _ShardedLogic
from tests.fake_engine import FakeEngine, _state
from tests.test_frontend_planner import build_circuit


def np_marginal(probs, qubits):
    """Reference marginal: bit j of the output index = qubit qubits[j]."""
    idx = np.arange(len(probs), dtype=np.int64)
    b = np.zeros_like(idx)
    for j, q in enumerate(qubits):
        b |= ((idx >> q) & 1) << j
    return np.bincount(b, weights=probs, minlength=1 << len(qubits))


def project_loop(indices, qubits):
    """Bit-by-bit Python restatement of a register's value."""
    out = []
    for k in np.asarray(indices).reshape(-1).tolist():
        v = 0
        for j, q in enumerate(qubits):
            if q is not None and (k >> q) & 1:
                v += 1 << j
        out.append(v)
    return np.asarray(out, dtype=np.int64).reshape(np.shape(indices))


class MarginalFakeEngine(FakeEngine):
    def __init__(self, device=0, dtype="complex128"):
        super().__init__(device, dtype)
        self.marginal_calls = 0

    def marginal_probabilities(self, plans, params, qubits):
        self.marginal_calls += 1
        rows = []
        for plan, vals in zip(plans, params):
            st = _state(self._plans[plan.plan_id], np.asarray(vals, dtype=np.float64).reshape(-1))
            rows.append(np_marginal(np.abs(st) ** 2, list(qubits)))
        return np.asarray(rows)


@pytest.fixture()
def fake_engines(monkeypatch):
    made = {}

    def get_engine(device=0, dtype="complex128"):
        return made.setdefault((device, dtype), MarginalFakeEngine(device, dtype))

    monkeypatch.setattr(pr, "get_engine", get_engine)
    monkeypatch.setattr(pr._native, "device_count", lambda: 3)
    return made


def case(n, layers, seed):
    genome, values = og.random_individual(n, layers, True, seed)
    instr = og.individual_circuit(genome, values)
    return instr, list(values), build_circuit(instr, n)


def assert_same_gates(measured, plain):
    """Measurements and barriers add no kernel op: the gate list is the unmeasured circuit's."""
    a, b = gl.from_circuit(measured), gl.from_circuit(plain)
    assert (a.n_qubits, a.n_params, a.param_names) == (b.n_qubits, b.n_params, b.param_names)
    assert a.ops == b.ops


# ---------------------------------------------------------------------------------------------- the circuit stand-in
def test_registers_of_the_stand_in():
    assert QuantumCircuit(3).cregs == [] and QuantumCircuit(3).num_clbits == 0 and QuantumCircuit(3).clbits == []
    assert QuantumCircuit(3, name="x").name == "x" and QuantumCircuit(3, "y").name == "y"
    assert QuantumCircuit(3, 0).cregs == []
    c = QuantumCircuit(3, 2)
    assert [(r.name, len(r)) for r in c.cregs] == [("c", 2)] and c.num_clbits == 2
    a, b = ClassicalRegister(2, "a"), ClassicalRegister(1, "b")
    c = QuantumCircuit(3, a, b)
    assert c.cregs == [a, b] and c.clbits == [a[0], a[1], b[0]] and all(isinstance(x, Clbit) for x in c.clbits)
    loc = c.find_bit(b[0])
    assert loc.index == 2 and loc.registers == [(b, 0)]
    assert c.find_bit(a[1]).index == 1 and c.find_bit(a[1]).registers == [(a, 1)]
    assert c.find_bit(c.qubits[2]).index == 2
    extra = ClassicalRegister(2, "e")
    c.add_register(extra)
    assert c.num_clbits == 5 and c.find_bit(extra[1]).index == 4
    with pytest.raises(ValueError, match="already exists"):
        c.add_register(ClassicalRegister(1, "a"))
    with pytest.raises(ValueError):
        c.find_bit(ClassicalRegister(1, "z")[0])


def measures(circ):
    return [(circ.find_bit(i.qubits[0]).index, circ.find_bit(i.clbits[0]).index) for i in circ.data if i.operation.name == "measure"]


def test_measure_broadcasts_like_qiskit():
    c = QuantumCircuit(3, 3)
    c.measure(range(3), range(3))
    assert measures(c) == [(0, 0), (1, 1), (2, 2)]
    c = QuantumCircuit(3, 3)
    c.measure(1, [0, 2])  # one qubit into several clbits
    c.measure([2, 0], c.cregs[0][:2])
    c.measure(c.qubits[1], c.clbits[1])
    assert measures(c) == [(1, 0), (1, 2), (2, 0), (0, 1), (1, 1)]
    reg = ClassicalRegister(2, "r")
    c = QuantumCircuit(2, reg)
    c.measure([0, 1], reg)
    assert measures(c) == [(0, 0), (1, 1)]
    with pytest.raises(ValueError, match="does not match"):
        QuantumCircuit(3, 2).measure([0, 1, 2], [0, 1])
    with pytest.raises(IndexError):
        QuantumCircuit(3, 2).measure(0, 5)


def test_copy_compose_and_measure_all_keep_registers():
    init = QuantumCircuit(3, 2)
    init.x(0)
    circ = QuantumCircuit(3)
    circ.h(1)
    circ.cx(1, 2)
    joined = init.compose(circ, inplace=False)
    assert [r.name for r in joined.cregs] == ["c"] and joined.clbits == init.clbits
    measured = joined.measure_all(inplace=False)
    assert [r.name for r in measured.cregs] == ["c", "meas"] and measured.num_clbits == 5
    assert [r.name for r in joined.cregs] == ["c"] and len(joined.data) == 3  # inplace=False leaves the original alone
    assert [r.name for r in measured.copy().cregs] == ["c", "meas"]
    assert [r.name for r in measured.decompose().cregs] == ["c", "meas"]
    assert measures(measured) == [(0, 2), (1, 3), (2, 4)]
    # an instruction's clbits map by index onto the destination's clbits
    src = QuantumCircuit(3, 2)
    src.measure(2, 1)
    dest = QuantumCircuit(3, ClassicalRegister(1, "x"), ClassicalRegister(2, "y"))
    out = dest.compose(src, clbits=[2, 0])
    assert measures(out) == [(2, 0)]
    assert gl.final_measurements(out) == [("x", 1, [2]), ("y", 2, [None, None])]
    with pytest.raises(ValueError, match="'out' edges"):
        QuantumCircuit(3).compose(src)
    # assign_parameters carries the registers
    _, values, pc = case(3, 2, 1)
    pc = QuantumCircuit(3, 1).compose(pc)
    pc.measure(1, 0)
    bound = pc.assign_parameters(values)
    assert [r.name for r in bound.cregs] == ["c"] and gl.final_measurements(bound) == [("c", 1, [1])]
    # measure_all twice: a second, fresh register
    twice = QuantumCircuit(2)
    twice.measure_all()
    twice.measure_all()
    assert [len(r) for r in twice.cregs] == [2, 2] and twice.cregs[1].name != "meas"
    # add_bits=False measures into the circuit's own first clbits
    own = QuantumCircuit(2, 3)
    own.measure_all(add_bits=False)
    assert gl.final_measurements(own) == [("c", 3, [0, 1, None])]
    with pytest.raises(ValueError):
        QuantumCircuit(3, 2).measure_all(add_bits=False)


# ---------------------------------------------------------------------------------------------- the measurement map
def measured_cases():
    """(description, circuit with measurements, the same circuit without them, expected map)."""
    _, _, base = case(5, 2, 7)
    out = []

    def add(desc, build, want):
        plain = base.copy()
        circ = QuantumCircuit(5, *build[0]).compose(base) if build[0] else base.copy()
        build[1](circ)
        out.append((desc, circ, plain, want))

    add("measure_all", ((), lambda c: c.measure_all()), [("meas", 5, [0, 1, 2, 3, 4])])
    add("QuantumCircuit(n, n)", ((5,), lambda c: c.measure(range(5), range(5))), [("c", 5, [0, 1, 2, 3, 4])])
    add("subset", ((2,), lambda c: c.measure([1, 3], [0, 1])), [("c", 2, [1, 3])])
    add("permuted clbits", ((3,), lambda c: c.measure([0, 2, 4], [2, 0, 1])), [("c", 3, [2, 4, 0])])
    add("one qubit into two clbits", ((2,), lambda c: c.measure(3, [0, 1])), [("c", 2, [3, 3])])
    add("clbit overwritten", ((2,), lambda c: (c.measure([0, 1], [0, 1]), c.measure(4, 0))), [("c", 2, [4, 1])])
    add("clbit never measured", ((3,), lambda c: c.measure([2, 1], [0, 2])), [("c", 3, [2, None, 1])])
    add("two registers", ((ClassicalRegister(2, "a"), ClassicalRegister(3, "b")), lambda c: c.measure([4, 0, 1, 2], [0, 2, 3, 4])),
        [("a", 2, [4, None]), ("b", 3, [0, 1, 2])])
    add("c next to meas", ((2,), lambda c: (c.measure([3, 4], [0, 1]), c.measure_all())), [("c", 2, [3, 4]), ("meas", 5, [0, 1, 2, 3, 4])])
    add("barrier after measure", ((1,), lambda c: (c.measure(2, 0), c.barrier(), c.measure(2, 0))), [("c", 1, [2])])
    add("gate on another qubit after measure", ((1,), lambda c: (c.measure(0, 0), c.x(1))), [("c", 1, [0])])
    return out


@pytest.mark.parametrize("desc", [c[0] for c in measured_cases()])
def test_final_measurements(desc):
    _, circ, plain, want = next(c for c in measured_cases() if c[0] == desc)
    assert gl.final_measurements(circ) == want
    if desc != "gate on another qubit after measure":
        assert_same_gates(circ, plain)


def test_final_measurements_without_registers():
    _, _, circ = case(4, 2, 3)
    assert gl.final_measurements(circ) == []
    assert pr._registers(circ) == [("meas", 4, [0, 1, 2, 3])]  # the read-out of a circuit without clbits, as before registers


def test_unsupported_measurements_raise():
    mid = QuantumCircuit(2, 2)
    mid.measure(0, 0)
    mid.h(0)
    with pytest.raises(NotImplementedError, match="mid-circuit measurement.*qubit 0"):
        gl.final_measurements(mid)
    mid2 = QuantumCircuit(3, 1)
    mid2.measure(1, 0)
    mid2.cx(0, 1)
    with pytest.raises(NotImplementedError, match="mid-circuit"):
        gl.final_measurements(mid2)
    reset = QuantumCircuit(2, 1)
    reset.append(Instruction("reset", 1), [0])
    reset.measure(0, 0)
    with pytest.raises(NotImplementedError, match="reset"):
        gl.final_measurements(reset)
    controlled = QuantumCircuit(2, 1)
    controlled.measure(0, 0)
    controlled.append(Instruction("x", 1), [1], [0])  # a gate reading a clbit
    with pytest.raises(NotImplementedError, match="classically controlled"):
        gl.final_measurements(controlled)
    flow = QuantumCircuit(2, 1)
    flow.append(Instruction("if_else", 1), [1])
    with pytest.raises(NotImplementedError, match="classically controlled"):
        gl.final_measurements(flow)
    conditioned = QuantumCircuit(2, 1)
    conditioned.x(0)
    conditioned.data[-1].operation._condition = (conditioned.clbits[0], 1)  # what c_if leaves on a Qiskit 1.x instruction
    with pytest.raises(NotImplementedError, match="classically controlled"):
        gl.final_measurements(conditioned)
    with pytest.raises(NotImplementedError):  # surfaced by the sampler's job
        pr.B200SamplerV2(seed=1).run([mid], shots=4).result()


# ---------------------------------------------------------------------------------------------- read-out of the shots
def test_register_values_against_a_bit_loop():
    rng = np.random.default_rng(4)
    k = rng.integers(0, 1 << 20, size=(3, 257))
    for qubits in ([0], [19], list(range(20)), [5, None, 3, 3, 17, None], [None, None], list(range(19, -1, -1)), [11, 4, 0, 9]):
        got = pr.register_values(k, qubits)
        assert got.shape == k.shape and np.array_equal(got, project_loop(k, qubits))
    assert np.array_equal(pr.register_values(k, list(range(20))), k)  # the identity map of measure_all
    with pytest.raises(NotImplementedError, match="63 bits"):
        pr.register_values(k, [0] * 64)


def test_join_data_order():
    a = ct.ShotRegister(np.array([1, 0, 3]), 2)
    b = ct.ShotRegister(np.array([0, 1, 1]), 1)
    c = ct.ShotRegister(np.array([5, 2, 7]), 3)
    res = ct.SamplerPubResult(ct.DataBin(a=a, b=b, c=c))
    joined = res.join_data()
    assert joined.num_bits == 6 and joined.indices.tolist() == [1 | 0 << 2 | 5 << 3, 0 | 1 << 2 | 2 << 3, 3 | 1 << 2 | 7 << 3]
    assert joined.get_bitstrings()[0] == "101" + "0" + "01"  # the first register is least significant: rightmost
    ba = res.join_data(["b", "a"])
    assert ba.num_bits == 3 and ba.indices.tolist() == [0 | 1 << 1, 1 | 0 << 1, 1 | 3 << 1]
    assert res.join_data(["c"]) is c
    with pytest.raises(ValueError):
        res.join_data([])
    shaped = ct.SamplerPubResult(ct.DataBin(a=ct.ShotRegister(np.arange(6).reshape(2, 3) % 4, 2, (2,)),
                                            b=ct.ShotRegister(np.ones((2, 3), dtype=np.int64), 1, (2,)), shape=(2,)))
    j = shaped.join_data()
    assert j.shape == (2,) and j.indices.tolist() == [[0 | 4, 1 | 4, 2 | 4], [3 | 4, 0 | 4, 1 | 4]]


@pytest.mark.parametrize("desc", ["subset", "permuted clbits", "one qubit into two clbits", "clbit overwritten", "clbit never measured",
                                  "two registers", "c next to meas", "measure_all"])
def test_run_projects_the_full_register_draws(fake_engines, desc):
    _, circ, plain, want = next(c for c in measured_cases() if c[0] == desc)
    _, values, _ = case(5, 2, 7)
    shots = 300
    res = pr.B200SamplerV2(seed=11).run([(circ, values)], shots=shots).result()[0]
    full = pr.B200SamplerV2(seed=11).sample_indices([plain], [values], shots)[0]
    assert list(res.data.keys()) == [name for name, _, _ in want]
    for name, size, qubits in want:
        reg = res.data[name]
        assert reg.num_bits == size and reg.num_shots == shots
        assert np.array_equal(reg.indices, project_loop(full, qubits))
        assert sum(reg.get_counts().values()) == shots and all(len(key) == size for key in reg.get_counts())
    if desc == "measure_all":
        assert np.array_equal(res.data.meas.indices, full)
    assert res.join_data().num_bits == sum(size for _, size, _ in want)


def test_run_with_a_parameter_array(fake_engines):
    _, values, base = case(4, 2, 9)
    circ = QuantumCircuit(4, ClassicalRegister(1, "x"), ClassicalRegister(2, "y")).compose(base)
    circ.measure([3, 0, 2], [0, 2, 1])
    rng = np.random.default_rng(2)
    pvals = np.asarray(values) + rng.normal(scale=0.3, size=(2, 3, len(values)))
    res = pr.B200SamplerV2(seed=3).run([(circ, pvals)], shots=50).result()[0]
    full = pr.B200SamplerV2(seed=3).sample_indices([base] * 6, list(pvals.reshape(6, -1)), 50).reshape(2, 3, 50)
    assert res.data.shape == (2, 3) and res.data.x.indices.shape == (2, 3, 50)
    assert np.array_equal(res.data.x.indices, project_loop(full, [3]))
    assert np.array_equal(res.data.y.indices, project_loop(full, [2, 0]))


def test_measured_circuits_keep_the_sampler_fast_path(fake_engines):
    """Measurements do not change the parsed gate list, so a measured and an unmeasured copy sample the same indices."""
    for desc, circ, plain, _ in measured_cases():
        if desc == "gate on another qubit after measure":
            continue
        _, values, _ = case(5, 2, 7)
        a = pr.B200SamplerV2(seed=2).sample_indices([circ], [values], 64)
        b = pr.B200SamplerV2(seed=2).sample_indices([plain], [values], 64)
        assert np.array_equal(a, b), desc


# ---------------------------------------------------------------------------------------------- marginal probabilities (host side)
def test_marginal_probabilities_routing_and_validation(fake_engines):
    smp = pr.B200SamplerV2(devices=[0, 1])
    cases = [case(6, 2, s) for s in range(4)]
    circuits, values = [c[2] for c in cases], [c[1] for c in cases]
    qubits = [4, 0, 5]
    got = smp.marginal_probabilities(circuits, values, qubits)
    assert got.shape == (4, 8) and got.dtype == np.float64
    for row, (instr, vals, _) in zip(got, cases):
        want = np_marginal(np.abs(oq.statevector(instr, 6, vals)) ** 2, qubits)
        assert np.allclose(row, want, atol=1e-13)
    assert sum(e.marginal_calls for e in fake_engines.values()) >= 1
    assert smp.marginal_probabilities([], [], [0]).shape == (0, 2)
    for bad, match in (([], "1 to 26"), (list(range(27)), "1 to 26"), ([1, 1], "distinct"), ([6], "distinct indices in \\[0, 6\\)"), ([-1], "distinct")):
        with pytest.raises(ValueError, match=match):
            smp.marginal_probabilities(circuits[:1], values[:1], bad)
    with pytest.raises(ValueError, match="same number of qubits"):
        smp.marginal_probabilities([circuits[0], case(5, 2, 0)[2]], [values[0], case(5, 2, 0)[1]], [0])
    with pytest.raises(ValueError, match="parameter vectors"):
        smp.marginal_probabilities(circuits, values[:2], [0])


class _NumpyShards(_ShardedLogic):
    """The sharded marginal's host logic over NumPy shards: each shard reduces its own amplitudes like ``qb_marginal_device``."""

    def __init__(self, physical, n_qubits, world, position):
        self._init_logic(n_qubits, world, 2)
        self.position = list(position)
        self.physical = physical

    def _marginal_parts(self, positions):
        size = 1 << self.n_local
        parts = []
        for r in range(self.world):
            k = np.arange(size, dtype=np.int64) | (r << self.n_local)
            p = np.abs(self.physical[r * size : (r + 1) * size]) ** 2
            b = np.zeros_like(k)
            for j, pos in enumerate(positions):
                b |= ((k >> pos) & 1) << j
            parts.append(np.bincount(b, weights=p, minlength=1 << len(positions)))
        return parts


@pytest.mark.parametrize("world", [2, 4])
def test_sharded_marginal_maps_logical_qubits(world):
    n = 8
    rng = np.random.default_rng(world)
    logical = rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)
    logical /= np.linalg.norm(logical)
    position = list(rng.permutation(n))
    # physical index: logical bit q at bit position[q]
    k = np.arange(1 << n)
    phys_of = np.zeros_like(k)
    for q in range(n):
        phys_of |= ((k >> q) & 1) << position[q]
    physical = np.empty_like(logical)
    physical[phys_of] = logical
    sv = _NumpyShards(physical, n, world, position)
    for qubits in ([0], [7], [6, 7], [7, 0, 3], list(range(n)), [position.index(n - 1), position.index(0)]):
        got = sv.marginal(qubits)
        assert np.allclose(got, np_marginal(np.abs(logical) ** 2, qubits), atol=1e-15)
    with pytest.raises(ValueError, match="distinct"):
        sv.marginal([0, 0])
