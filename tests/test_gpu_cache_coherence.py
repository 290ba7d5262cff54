"""The engine's cached evaluation state against fresh evaluations, across plan, Hamiltonian and batch lifetimes.

Most values an optimizer loop consumes come from cached state rather than from a fresh kernel chain: the single-circuit CUDA
graphs keyed by (plan, Hamiltonian, copies), the one-shot batch re-used for an identical list, the cached prefix states, the
resident batches and the structural plan cache.  These tests interleave evaluations with compiles, destroys, re-prefixing,
evictions, workspace and index-width changes, and check every value against the float64 oracle (NumPy below 16 qubits, the C
oracle from 16 on): ``|got - ref| / max(1, |ref|) <= 1e-10`` for expectation values, the sampler tests' "<= 1 flip to a
neighbouring or non-zero state" rule for shots, ``assert_cvar`` for CVaR.  Every tenth step of the sequence test is also
replayed on a freshly created engine, where the same call runs the same launch shape cold and must give the same bits.
"""
import ctypes
import gc
import math

import numpy as np
import pytest

from oracle import c_oracle
from oracle import evqe_genome as og
from oracle import qiskit_semantics as oq
from queasars_b200 import _native
from queasars_b200 import gate_list as gl
from queasars_b200.circuit import QuantumCircuit
from queasars_b200.operators import SparsePauliOp
from tests.test_frontend_planner import build_circuit
from tests.test_gpu_cvar_exact import assert_cvar
from tests.test_gpu_parity import random_ising, tfim

pytestmark = pytest.mark.gpu

TOL = 1e-10


def Engine(**kw):
    from queasars_b200.engine import Engine as _Engine

    return _Engine(device=0, dtype="complex128", **kw)


def assert_value(got, want, what):
    err = abs(got - want) / max(1.0, abs(want))
    assert err <= TOL, f"{what}: got {got!r}, oracle {want!r} (rel {err:.2e})"


# ------------------------------------------------------------------------------------ oracle-side model objects
class Circ:
    """An EVQE individual: oracle instructions, parameter rows and the gate list the engine compiles.  ``parameterized``:
    the layers that keep named parameters ({-1}: the leading layers are bound, the prefix-reuse pattern)."""

    def __init__(self, n, layers, seed, parameterized=None):
        genome, values = og.random_individual(n, layers, True, seed)
        self.n = n
        self.instr = og.individual_circuit(genome, values, parameterized)
        if parameterized is not None:
            (lid,) = parameterized
            values = values[og.layer_value_slice(genome, lid)]
        self.gates = gl.from_circuit(build_circuit(self.instr, n))
        rng = np.random.default_rng(seed + 17)
        self.rows = [list(values)] + [list(rng.uniform(0, 2 * math.pi, len(values))) for _ in range(2)]
        self._states = {}

    def state(self, r):
        if r not in self._states:
            if self.n < 16:
                self._states[r] = oq.statevector(self.instr, self.n, self.rows[r])
            else:
                self._states[r] = c_oracle.evaluate(self.instr, self.n, self.rows[r], None, np.empty(1 << self.n, dtype=np.complex128))[1]
        return self._states[r]


def pauli_terms(n, seed):
    """TFIM plus a few random X / Y / Z strings with complex coefficients (non-diagonal)."""
    rng = np.random.default_rng(seed)
    terms = tfim(n)
    for _ in range(3):
        terms.append(("".join(rng.choice(list("IXYZ"), size=n)), complex(rng.normal(), rng.normal())))
    return terms


class Op:
    """A Hamiltonian of the model: diagonal (random Ising) or a Pauli sum, with its oracle value of a state."""

    def __init__(self, n, diagonal, seed, build_table=None):
        self.n, self.diagonal, self.build_table = n, diagonal, build_table
        self.terms = random_ising(n, seed) if diagonal else pauli_terms(n, seed)
        self.op = SparsePauliOp.from_list(self.terms)
        self._table = None

    @property
    def table(self):
        if self._table is None:
            diag = oq.diag_terms_from_labels(self.terms)
            self._table = oq.diagonal_table(self.n, diag) if self.n < 16 else c_oracle.diag_table(self.n, diag)
        return self._table

    def value(self, state):
        if self.diagonal:
            return float(np.dot(state.real**2 + state.imag**2, self.table))
        return oq.estimator_expectation(state, self.terms) if self.n < 16 else c_oracle.pauli_sum(state, self.n, self.terms)

    def make(self, engine):
        return engine.hamiltonian(self.op, build_table=self.build_table)


def compile_plan(engine, circ, kind, probs_only):
    """kind "shared": through the structural plan cache; "own": a plan of its own (destroyed with its handle); "prefix":
    ``compile_with_prefix_reuse`` (falls back to ``compile`` when there is no constant prefix)."""
    if kind == "prefix":
        return engine.compile_with_prefix_reuse(circ.gates, drop_final_phases=probs_only)
    return engine.compile(circ.gates, cache=kind == "shared", drop_final_phases=probs_only)


class ObsSet:
    """Observables of one width evaluated together (``Engine.observables``)."""

    def __init__(self, ops, engine):
        self.ops, self.diagonal = ops, all(o.diagonal for o in ops)
        self.handle = engine.observables([o.op for o in ops])


class Plan:
    def __init__(self, engine, circ, kind, probs_only):
        self.circ, self.kind, self.probs_only = circ, kind, probs_only
        self.handle = compile_plan(engine, circ, kind, probs_only)


# ------------------------------------------------------------------------------------ calls: run on any engine, check against the oracle
class Call:
    """One evaluation: ``route``, the model plans, their parameter row ids, and the operator / observables / extra arguments.
    ``run(engine, plan_of, ham_of, batch_of)`` performs it on an engine, mapping model objects to that engine's handles."""

    def __init__(self, route, plans, rows, op=None, obs=None, extra=None):
        self.route, self.plans, self.rows, self.op, self.obs, self.extra = route, plans, rows, op, obs, extra

    def params(self):
        return [p.circ.rows[r] for p, r in zip(self.plans, self.rows)]

    def run(self, engine, plan_of, ham_of, obs_of, batch_of):
        handles = [plan_of(p) for p in self.plans]
        params = self.params()
        if self.route == "exp":
            return engine.expectation(handles, params, ham_of(self.op))
        if self.route == "submit":
            count = engine.expectation_submit(handles, params, ham_of(self.op))
            return engine.expectation_collect(count)
        if self.route == "resident":
            rb = batch_of(self)
            rb.set_params(params)
            rb.run()
            return rb.read()
        if self.route == "sample":
            return engine.sample(handles, params, self.extra.shape[1], self.extra)
        if self.route == "cvar":
            return engine.cvar(handles, params, ham_of(self.op), self.extra)
        if self.route == "many":
            return engine.expectation_many(handles, params, obs_of(self.obs))
        if self.route == "sv":
            return engine.statevector(handles[0], params[0])
        raise ValueError(self.route)

    def check(self, got, step):
        states = [p.circ.state(r) for p, r in zip(self.plans, self.rows)]
        what = f"step {step} {self.route}"
        if self.route in ("exp", "submit", "resident"):
            assert len(got) == len(states)
            for i, (g, st) in enumerate(zip(got, states)):
                assert_value(g, self.op.value(st), f"{what} entry {i}")
        elif self.route == "sample":
            for row, st in enumerate(states):
                n = self.plans[row].circ.n
                want = oq.sample_indices(st, self.extra.shape[1], uniforms=self.extra[row]) if n < 16 else c_oracle.sample_indices(st, n, self.extra[row])
                mismatches = np.nonzero(got[row] != want)[0]
                assert len(mismatches) <= 1, f"{what} row {row}: {len(mismatches)} indices differ"
                for i in mismatches:  # only a flip to an adjacent state at a CDF boundary
                    assert abs(int(got[row][i]) - int(want[i])) <= 1 or abs(st[got[row][i]]) ** 2 > 0, what
        elif self.route == "cvar":
            for g, st in zip(got, states):
                assert_cvar(g, st.real**2 + st.imag**2, self.op.table, self.extra, TOL)
        elif self.route == "many":
            ops = self.obs.ops
            assert got.shape == (len(states), len(ops))
            for i, st in enumerate(states):
                for j, op in enumerate(ops):
                    assert_value(got[i, j], op.value(st), f"{what} entry {i} observable {j}")
        elif self.route == "sv":
            err = float(np.max(np.abs(got - states[0])))
            assert err <= 1e-12, f"{what}: max amplitude error {err:.2e}"


def replay_cold(call, workspace_limit, index_bits):
    """The same call on a freshly created engine (same workspace limit and index width, so the same launch shape)."""
    fresh = Engine(workspace_limit=workspace_limit)
    try:
        if index_bits == 64:
            fresh.set_index_width(64)
        plans, hams, obs = {}, {}, {}

        def plan_of(p):
            if id(p) not in plans:
                plans[id(p)] = compile_plan(fresh, p.circ, p.kind, p.probs_only)
            return plans[id(p)]

        def ham_of(op):
            if id(op) not in hams:
                hams[id(op)] = op.make(fresh)
            return hams[id(op)]

        def obs_of(o):
            if id(o) not in obs:
                obs[id(o)] = fresh.observables([op.op for op in o.ops])
            return obs[id(o)]

        def batch_of(c):
            return fresh.resident_batch([plan_of(p) for p in c.plans], ham_of(c.op))

        return call.run(fresh, plan_of, ham_of, obs_of, batch_of)
    finally:
        fresh.close()


# ------------------------------------------------------------------------------------ the model-based sequence
WIDTHS = {0: (8, 12), 1: (10, 14), 2: (9, 16)}
WIDE = 20
STEPS = 150
VALUE_ROUTES = ("single", "batch", "submit", "resident", "sample", "cvar", "many", "sv")


class Model:
    def __init__(self, engine, seed):
        self.engine, self.rng, self.seed = engine, np.random.default_rng(seed), seed
        self.widths = WIDTHS[seed]
        self.pool = {n: [Circ(n, 2 + k % 3, 1000 * seed + 20 * n + k, {-1} if k % 2 else None) for k in range(6)] for n in self.widths}
        self.pool[WIDE] = [Circ(WIDE, 2, 1000 * seed + 900 + k) for k in range(2)]
        self.plans, self.ops, self.obs, self.batches = [], [], [], []
        self.index_bits = 32
        self.counts: dict = {}

    # -- model upkeep
    def new_plan(self, n, probs_only=None):
        circ = self.pool[n][int(self.rng.integers(len(self.pool[n])))]
        kind = ("shared", "own", "prefix")[int(self.rng.integers(3))]
        if probs_only is None:
            probs_only = bool(self.rng.random() < 0.3)
        plan = Plan(self.engine, circ, kind, probs_only)
        self.plans.append(plan)
        return plan

    def new_op(self, n, diagonal=None):
        diagonal = bool(self.rng.random() < 0.6) if diagonal is None else diagonal
        op = Op(n, diagonal, int(self.rng.integers(1 << 20)), build_table=(None, False)[int(self.rng.integers(2))])
        op.handle = op.make(self.engine)
        self.ops.append(op)
        return op

    def op_for(self, n, diagonal=None):
        cands = [o for o in self.ops if o.n == n and (diagonal is None or o.diagonal == diagonal)]
        return cands[int(self.rng.integers(len(cands)))] if cands and self.rng.random() < 0.8 else self.new_op(n, diagonal)

    def plans_for(self, n, count, diagonal):
        """``count`` plans (repetition allowed) of width ``n`` that may be evaluated against a (non-)diagonal operator: a plan
        that drops its final phases gives |psi|^2 only."""
        cands = [p for p in self.plans if p.circ.n == n and (diagonal or not p.probs_only)]
        while len(cands) < 3:
            cands.append(self.new_plan(n, probs_only=False if not diagonal else None))
        return [cands[int(i)] for i in self.rng.integers(len(cands), size=count)]

    def rows(self, count):
        return [int(r) for r in self.rng.integers(3, size=count)]

    # -- steps
    def step(self, i):
        n = WIDE if i in (40, 110) else self.widths[int(self.rng.integers(len(self.widths)))]
        if n == WIDE:
            kind = ("single", "batch", "cvar")[int(self.rng.integers(3))]
        elif i % 10 == 9:
            kind = VALUE_ROUTES[int(self.rng.integers(len(VALUE_ROUTES)))]
        else:
            kinds = ["compile", "drop", "new_ham", "index"] + list(VALUE_ROUTES) * 2
            kind = kinds[int(self.rng.integers(len(kinds)))]
        self.counts[kind] = self.counts.get(kind, 0) + 1
        if kind == "compile":
            self.new_plan(n)
            return None
        if kind == "drop":
            pools = [lst for lst in (self.plans, self.ops, self.obs, self.batches) if lst]
            if pools:
                lst = pools[int(self.rng.integers(len(pools)))]
                lst.pop(int(self.rng.integers(len(lst))))
                gc.collect()
            return None
        if kind == "new_ham":
            self.new_op(n)
            return None
        if kind == "index":
            self.index_bits = 96 - self.index_bits
            self.engine.set_index_width(self.index_bits)
            return None
        return getattr(self, "call_" + kind)(n)

    def call_single(self, n):
        op = self.op_for(n)
        (plan,) = self.plans_for(n, 1, op.diagonal)
        copies = int(self.rng.integers(1, 5))
        return [Call("exp", [plan] * copies, self.rows(copies), op=op)]

    def call_batch(self, n):
        op = self.op_for(n)
        count = int(self.rng.integers(2, 4)) if n == WIDE else int(self.rng.integers(5, 41))
        plans = self.plans_for(n, count, op.diagonal)
        rows = self.rows(count)
        first = Call("exp", plans, rows, op=op)
        # the identical list again (the assembled one-shot batch is re-used as it is), then with other parameter rows
        return [first, Call("exp", plans, rows, op=op), Call("exp", plans, self.rows(count), op=op)]

    def call_submit(self, n):
        op = self.op_for(n)
        count = int(self.rng.integers(5, 41))
        return [Call("submit", self.plans_for(n, count, op.diagonal), self.rows(count), op=op)]

    def call_resident(self, n):
        live = [b for b in self.batches if b[1][0].circ.n == n]
        if live and self.rng.random() < 0.6:
            _, plans, op = entry = live[int(self.rng.integers(len(live)))]
        else:
            op = self.op_for(n)
            plans = self.plans_for(n, int(self.rng.integers(2, 9)), op.diagonal)
            entry = (self.engine.resident_batch([p.handle for p in plans], op.handle), plans, op)
            self.batches.append(entry)
        call = Call("resident", plans, self.rows(len(plans)), op=op)
        call.batch = entry[0]
        return [call]

    def call_sample(self, n):
        count = int(self.rng.integers(1, 7))
        plans = self.plans_for(n, count, True)
        return [Call("sample", plans, self.rows(count), extra=self.rng.random((count, 256)))]

    def call_cvar(self, n):
        op = self.op_for(n, diagonal=True)
        count = int(self.rng.integers(1, 9)) if n != WIDE else 2
        alpha = (0.1, 0.5, 1.0)[int(self.rng.integers(3))]
        return [Call("cvar", self.plans_for(n, count, True), self.rows(count), op=op, extra=alpha)]

    def call_many(self, n):
        live = [o for o in self.obs if o.ops[0].n == n]
        if live and self.rng.random() < 0.6:
            obs = live[int(self.rng.integers(len(live)))]
        else:
            diagonal = bool(self.rng.random() < 0.5)  # all diagonal, or a mix
            ops = [Op(n, diagonal or bool(self.rng.random() < 0.5), int(self.rng.integers(1 << 20))) for _ in range(int(self.rng.integers(2, 4)))]
            obs = ObsSet(ops, self.engine)
            self.obs.append(obs)
        count = int(self.rng.integers(1, 9))
        return [Call("many", self.plans_for(n, count, obs.diagonal), self.rows(count), obs=obs)]

    def call_sv(self, n):
        return [Call("sv", self.plans_for(n, 1, False), self.rows(1))]


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_model_based_sequence(seed):
    engine = Engine()
    model = Model(engine, seed)
    replays = 0
    for i in range(STEPS):
        calls = model.step(i)
        if not calls:
            continue
        last = None
        for call in calls:
            got = call.run(engine, lambda p: p.handle, lambda op: op.handle, lambda o: o.handle, lambda c: c.batch)
            call.check(got, i)
            if last is not None and call.rows == last[0].rows:
                assert np.array_equal(got, last[1]), f"step {i}: the identical call again gave other bits"
            last = (call, got)
        if i % 10 == 9:
            call, got = last
            cold = replay_cold(call, 0, model.index_bits)
            assert np.array_equal(np.asarray(got), np.asarray(cold)), f"step {i} {call.route}: cached and cold evaluations differ"
            replays += 1
    assert replays == STEPS // 10
    for route in ("compile", "drop", "single", "batch", "resident"):
        assert model.counts.get(route, 0) > 0, (route, model.counts)
    engine.close()


# ------------------------------------------------------------------------------------ eviction of single-circuit graphs
def test_graph_eviction_by_bytes():
    # workspace 64 MiB: the graph budget is min(4 GiB, 64 MiB / 8) = 8 MiB and a call is graphed while its states take at most a
    # quarter of it, 2 MiB.  At 16 qubits complex128 a copy is 1 MiB: 1 and 2 copies are graphed, 3 copies run without a graph;
    # eight one-copy graphs fill the budget and the ninth distinct one evicts the least recently used.
    engine = Engine(workspace_limit=64 << 20)
    n = 16
    circs = [Circ(n, 2, 500 + k) for k in range(10)]
    op = Op(n, True, 41)
    ham = op.make(engine)
    plans = [engine.compile(c.gates, cache=False) for c in circs]
    for rnd in range(2):  # second round: the first graphs were evicted and are captured again
        for k, (plan, circ) in enumerate(zip(plans, circs)):
            r = (k + rnd) % 3
            assert_value(engine.expectation([plan], [circ.rows[r]], ham)[0], op.value(circ.state(r)), f"round {rnd} plan {k}")
        for copies in (2, 3):
            got = engine.expectation([plans[rnd]] * copies, [circs[rnd].rows[r] for r in range(copies)], ham)
            for r in range(copies):
                assert_value(got[r], op.value(circs[rnd].state(r)), f"round {rnd}, {copies} copies, entry {r}")
    engine.close()


def test_graph_eviction_by_count():
    """260 distinct (plan, Hamiltonian, copies) keys pass the limit of 256 cached graphs; the first keys, evicted, are
    captured again and still give the oracle's values."""
    engine = Engine()
    n = 8
    circs = [Circ(n, 3, 600 + k) for k in range(5)]
    op = Op(n, False, 43)
    ham = op.make(engine)
    plans = [(engine.compile(circs[k % 5].gates, cache=False), circs[k % 5]) for k in range(65)]
    keys = [(plan, circ, copies) for plan, circ in plans for copies in (1, 2, 3, 4)]
    assert len(keys) == 260

    def check(plan, circ, copies, what):
        rows = [(copies + r) % 3 for r in range(copies)]
        got = engine.expectation([plan] * copies, [circ.rows[r] for r in rows], ham)
        for g, r in zip(got, rows):
            assert_value(g, op.value(circ.state(r)), what)

    for k, key in enumerate(keys):
        check(*key, f"key {k}")
    for k, key in enumerate(keys[:24]):
        check(*key, f"key {k} again")
    engine.close()


# ------------------------------------------------------------------------------------ directed: prefix set after a graph exists
def split_prefix(gates):
    split = next(i for i, op in enumerate(gates.ops) if any(a.slot >= 0 or a.slot2 >= 0 for a in op.angles))
    prefix = gl.GateList(gates.n_qubits, list(gates.ops[:split]), 0, ())
    suffix = gl.GateList(gates.n_qubits, list(gates.ops[split:]), gates.n_params, gates.param_names)
    return prefix, suffix


def suffix_state(suffix_gates, values):
    """The suffix alone applied to |0...0> (what a plan without its prefix computes), by the NumPy gate-list emulator."""
    from tests.fake_engine import _state

    return _state(suffix_gates, values)


def test_set_prefix_after_a_graph_was_cached():
    """A plan compiled for an existing state is evaluated through the single-circuit graph path (from |0...0>), then given a
    prefix over the C-ABI: the next one-circuit call must start from the prefix state -- prefix and suffix together, i.e. the
    whole circuit.  The same through a resident batch, whose parameters, uploaded before, stay valid."""
    engine = Engine()
    lib, ctx = engine._lib, engine._ctx
    circ = Circ(12, 4, 71, {-1})
    op = Op(12, True, 5)
    ham = op.make(engine)
    pre_gates, suf_gates = split_prefix(circ.gates)
    prefix = engine.compile(pre_gates, from_zero_state=True, cache=False, defer=False)
    for route in ("graph", "resident"):
        suffix = engine.compile(suf_gates, from_zero_state=False, cache=False, defer=False)
        if route == "graph":
            for copies in (1, 2):
                got = engine.expectation([suffix] * copies, circ.rows[:copies], ham)
                for r in range(copies):
                    assert_value(got[r], op.value(suffix_state(suf_gates, circ.rows[r])), f"suffix alone, {copies} copies")
            _native.check(lib.qb_plan_set_prefix(ctx, suffix.plan_id, prefix.plan_id))
            suffix.prefix = prefix
            for copies in (1, 2):
                got = engine.expectation([suffix] * copies, circ.rows[1 : 1 + copies], ham)
                for r in range(copies):
                    assert_value(got[r], op.value(circ.state(1 + r)), f"graph path after qb_plan_set_prefix, {copies} copies")
        else:
            rb = engine.resident_batch([suffix] * 3, ham)
            rb.set_params(circ.rows)
            rb.run()
            for r, g in enumerate(rb.read()):
                assert_value(g, op.value(suffix_state(suf_gates, circ.rows[r])), "resident batch, suffix alone")
            _native.check(lib.qb_plan_set_prefix(ctx, suffix.plan_id, prefix.plan_id))
            suffix.prefix = prefix
            rb.run()  # the parameters uploaded before the prefix was set
            for r, g in enumerate(rb.read()):
                assert_value(g, op.value(circ.state(r)), "resident batch after qb_plan_set_prefix")
            rb.set_params(circ.rows[::-1])
            rb.run()
            for r, g in enumerate(rb.read()):
                assert_value(g, op.value(circ.state(2 - r)), "resident batch after qb_plan_set_prefix, new parameters")
            rb.close()
    engine.close()


# ------------------------------------------------------------------------------------ directed: resident batch with a destroyed member
@pytest.mark.parametrize("gone", ["plan", "hamiltonian"])
def test_resident_batch_with_a_destroyed_member_is_refused(gone):
    """A resident batch whose plan or Hamiltonian was destroyed is re-validated before anything runs: every entry point
    returns QB_ERR_NOT_FOUND and launches nothing.  qb_batch_set_params is asserted first -- it touches the batch's own
    buffers only -- so that a library without the check fails here, before a launch against freed memory."""
    engine = Engine()
    lib, ctx = engine._lib, engine._ctx
    n = 10
    circs = [Circ(n, 3, 80 + k) for k in range(3)]
    op = Op(n, True, 9)
    ham = op.make(engine)
    plans = [engine.compile(c.gates, cache=False) for c in circs]
    unrelated = engine.compile(circs[0].gates, cache=False)
    ids = np.array([p.plan_id for p in plans], dtype=np.int64)
    batch_id = ctypes.c_int64()
    _native.check(lib.qb_batch_create(ctx, len(plans), _native.ptr(ids), ham.ham_id, ctypes.byref(batch_id)))
    batch_id = batch_id.value
    flat = np.concatenate([np.asarray(c.rows[1]) for c in circs])
    offsets = np.concatenate([[0], np.cumsum([len(c.rows[1]) for c in circs])]).astype(np.int64)
    out = np.empty(len(plans))

    def run_and_read():
        _native.check(lib.qb_batch_set_params(ctx, batch_id, _native.ptr(flat), _native.ptr(offsets)))
        _native.check(lib.qb_batch_run(ctx, batch_id))
        _native.check(lib.qb_batch_read(ctx, batch_id, _native.ptr(out)))
        for g, c in zip(out, circs):
            assert_value(g, op.value(c.state(1)), "resident batch")

    run_and_read()
    _native.check(lib.qb_plan_destroy(ctx, unrelated.plan_id))  # another plan goes: the batch is re-assembled, same values
    run_and_read()
    if gone == "plan":
        _native.check(lib.qb_plan_destroy(ctx, plans[1].plan_id))
    else:
        _native.check(lib.qb_hamiltonian_destroy(ctx, ham.ham_id))
    before = engine.launch_count
    assert lib.qb_batch_set_params(ctx, batch_id, _native.ptr(flat), _native.ptr(offsets)) == _native.QB_ERR_NOT_FOUND
    assert lib.qb_batch_run(ctx, batch_id) == _native.QB_ERR_NOT_FOUND
    ms, states, count = np.zeros(64, dtype=np.float32), np.zeros(64, dtype=np.int32), ctypes.c_int()
    assert lib.qb_batch_run_timed(ctx, batch_id, 64, _native.ptr(ms), _native.ptr(states), ctypes.byref(count)) == _native.QB_ERR_NOT_FOUND
    assert lib.qb_batch_read(ctx, batch_id, _native.ptr(out)) == _native.QB_ERR_NOT_FOUND
    assert engine.launch_count == before
    assert lib.qb_batch_run(ctx, batch_id) == _native.QB_ERR_NOT_FOUND  # and stays refused
    _native.check(lib.qb_batch_destroy(ctx, batch_id))
    engine.close()


# ------------------------------------------------------------------------------------ directed: prefix destroyed, suffix lives
def test_prefix_plan_destroyed_while_its_suffix_lives():
    """The suffix keeps the prefix state it computed: its values stay right on the graph and the batch paths.  A suffix that
    never computed it cannot start any more and says so."""
    engine = Engine()
    lib, ctx = engine._lib, engine._ctx
    circ = Circ(13, 4, 91, {-1})
    op = Op(13, False, 12)
    ham = op.make(engine)
    pre_gates, suf_gates = split_prefix(circ.gates)
    prefix = engine.compile(pre_gates, from_zero_state=True, cache=False, defer=False)
    used, unused = (engine.compile(suf_gates, from_zero_state=False, cache=False, defer=False) for _ in range(2))
    for s in (used, unused):
        _native.check(lib.qb_plan_set_prefix(ctx, s.plan_id, prefix.plan_id))
    assert_value(engine.expectation([used], [circ.rows[0]], ham)[0], op.value(circ.state(0)), "before")
    _native.check(lib.qb_plan_destroy(ctx, prefix.plan_id))
    for copies in (1, 2, 5):
        got = engine.expectation([used] * copies, [circ.rows[r % 3] for r in range(copies)], ham)
        for r, g in enumerate(got):
            assert_value(g, op.value(circ.state(r % 3)), f"after the prefix was destroyed, {copies} copies")
    with pytest.raises(_native.QbError) as err:
        engine.expectation([unused], [circ.rows[0]], ham)
    assert err.value.code == _native.QB_ERR_NOT_FOUND
    engine.close()


# ------------------------------------------------------------------------------------ Python-side caches
def test_prefix_budget_overflow_falls_back_to_compile(monkeypatch):
    """QB_PREFIX_CACHE_MB=1 holds four 14-qubit prefix states (256 KiB each): the fifth circuit is compiled whole, and a
    released handle gives its share of the budget back."""
    monkeypatch.setenv("QB_PREFIX_CACHE_MB", "1")
    engine = Engine()
    n = 14
    circs = [Circ(n, 4, 300 + k, {-1}) for k in range(6)]
    op = Op(n, True, 3)
    ham = op.make(engine)
    handles = [engine.compile_with_prefix_reuse(c.gates) for c in circs[:5]]
    assert [h.prefix is not None for h in handles] == [True] * 4 + [False]

    def check(hs, cs, what):
        got = engine.expectation(hs, [c.rows[1] for c in cs], ham)
        for k, (g, c) in enumerate(zip(got, cs)):
            assert_value(g, op.value(c.state(1)), f"{what} entry {k}")
        for h, c in zip(hs, cs):
            assert_value(engine.expectation([h], [c.rows[2]], ham)[0], op.value(c.state(2)), f"{what} single")

    check(handles, circs[:5], "budget full")
    del handles[0]
    gc.collect()
    handles.append(engine.compile_with_prefix_reuse(circs[5].gates))
    assert handles[-1].prefix is not None
    check(handles, circs[1:6], "budget released")
    engine.close()


def test_plan_cache_overflow_keeps_live_handles():
    """More than 4096 distinct structures clear the structural plan cache; handles held across the clear stay valid, and the
    same structure compiled after it is a new plan with the same values."""
    engine = Engine()
    n = 3
    op = Op(n, True, 7)
    ham = op.make(engine)

    def circuit(k):
        theta = 0.001 * (k + 1)
        instr = [("h", (0,), ()), ("h", (1,), ()), ("rz", (1,), (theta,)), ("h", (1,), ()), ("cx", (0, 2), ())]
        circ = QuantumCircuit(n)
        circ.h(0), circ.h(1), circ.rz(theta, 1), circ.h(1), circ.cx(0, 2)
        return instr, gl.from_circuit(circ)

    kept = {}
    for k in range(4100):
        instr, gates = circuit(k)
        handle = engine.compile(gates)
        if k % 512 == 0 or k >= 4090:
            kept[k] = (handle, instr, gates)
    assert len(engine._plan_cache) < 4096  # the cache was cleared on the way
    ks = sorted(kept)
    got = engine.expectation([kept[k][0] for k in ks], [[] for _ in ks], ham)
    for k, g in zip(ks, got):
        assert_value(g, op.value(oq.statevector(kept[k][1], n)), f"structure {k}")
    again = engine.compile(kept[0][2])
    assert again is not kept[0][0] and again.plan_id != kept[0][0].plan_id
    assert_value(engine.expectation([again], [[]], ham)[0], op.value(oq.statevector(kept[0][1], n)), "recompiled after the clear")
    assert_value(engine.expectation([kept[0][0]], [[]], ham)[0], op.value(oq.statevector(kept[0][1], n)), "held across the clear")
    engine.close()


def test_lowered_workspace_limit_chunks_a_reused_list():
    """An identical list evaluated again after the workspace limit was lowered must be cut into chunks (the assembled
    batch is not re-used whole); with the limit restored it runs in one piece again, bit for bit as before."""
    engine = Engine()
    lib, ctx = engine._lib, engine._ctx
    n = 14
    circs = [Circ(n, 3, 400 + k) for k in range(12)]
    op = Op(n, False, 21)
    ham = op.make(engine)
    plans = [engine.compile(c.gates) for c in circs]
    rows = [c.rows[k % 3] for k, c in enumerate(circs)]

    def check(got, what):
        for k, (g, c) in enumerate(zip(got, circs)):
            assert_value(g, op.value(c.state(k % 3)), f"{what} entry {k}")

    first = engine.expectation(plans, rows, ham)
    check(first, "whole")
    assert np.array_equal(engine.expectation(plans, rows, ham), first)
    state_bytes = 16 << n
    _native.check(lib.qb_context_set_workspace_limit(ctx, 4 * state_bytes))  # four states per chunk
    check(engine.expectation(plans, rows, ham), "four per chunk")
    check(engine.expectation(plans[:5], rows[:5], ham), "four per chunk, shorter list")
    _native.check(lib.qb_context_set_workspace_limit(ctx, 0))
    assert np.array_equal(engine.expectation(plans, rows, ham), first)
    engine.close()
