"""Every dispatch class of the sweep kernel on the GPU, against the plan emulator (the same encoded program executed in NumPy)
and the oracle: all six kernel builds, widths from one tile to 20 qubits, zero / partial / full product starts and cached
prefix states, tiles per CTA and batch composition, the launch switches (bit-identical to the default engine), rank offsets
of sharded segments, and the sampler at the edges of its CDF.  tests/test_dispatch_coverage.py checks on the CPU that the
circuits used here reach every body class."""
import functools
import math

import numpy as np
import pytest

from oracle import qiskit_semantics as oq
from queasars_b200 import gate_list as gl
from queasars_b200.operators import SparsePauliOp
from tests import dispatch_coverage as dc
from tests.plan_emulator import run_program
from tests.test_gpu_parity import random_ising, rel_err, tfim

pytestmark = pytest.mark.gpu

VARIANTS = ["c128", "c64", "tile12", "reg3", "idx64", "c64_idx64"]
WIDTHS = [11, 12, 13, 14, 15, 16]


def make_engine(kind="c128"):
    from queasars_b200.engine import Engine

    kw = {"c64": {"dtype": "complex64"}, "c64_idx64": {"dtype": "complex64"}, "tile12": {"tile_bits": 12}, "reg3": {"reg_bits": 3}}.get(kind, {})
    eng = Engine(device=0, **kw)
    if kind.endswith("idx64"):
        eng.set_index_width(64)
    return eng


@functools.lru_cache(maxsize=None)
def case(n, label, tile_bits):
    """(instructions, parameter values, gate list, oracle statevector) of one family member."""
    fam = dict(dc.circuit_family(n, tile_bits, seed=n, n_random=1 if n > 16 else 2))
    fam["zero"] = dc.zero_start_circuit(n, 3 * n)
    instr = fam[label]
    values = dc.values_for(instr, 7 * n + len(label))
    return instr, values, dc.gates_of(instr, n), oq.statevector(instr, n, values)


def labels(n, tile_bits):
    return [lab for lab, _ in dc.circuit_family(n, tile_bits, seed=n, n_random=1 if n > 16 else 2)]


@functools.lru_cache(maxsize=None)
def emulated(n, label, tile_bits, reg_bits, drop, from_zero_state=True):
    _, values, gates, _ = case(n, label, tile_bits)
    _, enc = dc.plan_for(gates, tile_bits, reg_bits, drop, from_zero_state)
    return run_program(enc, max(n, tile_bits), tile_bits, values, reg_bits=reg_bits)[: 1 << n]


@functools.lru_cache(maxsize=None)
def hamiltonians(n):
    diag = random_ising(n, 100 + n)
    rng = np.random.default_rng(n)
    mixed = tfim(n) + [("".join(rng.choice(list("IXYZ"), size=n)), complex(rng.normal(), rng.normal())) for _ in range(4)]
    return diag, oq.diagonal_table(n, oq.diag_terms_from_labels(diag)), mixed


# ------------------------------------------------------------------------------------ a. every engine variant
@pytest.mark.parametrize("kind", VARIANTS)
def test_every_dispatch_class_on_every_kernel_build(kind):
    eng = make_engine(kind)
    single = eng.dtype == "complex64"
    K, R = eng.tile_bits, eng.reg_bits
    tol_sv, tol_ev = (2e-6, 1e-4) if single else (1e-13, 1e-10)
    cov, cov_drop = dc.Coverage(R), dc.Coverage(R)
    for n in WIDTHS + [20]:
        diag, table, mixed = hamiltonians(n)
        ham_d, ham_x = eng.hamiltonian(SparsePauliOp.from_list(diag)), eng.hamiltonian(SparsePauliOp.from_list(mixed))
        labs = labels(n, K) if n <= 16 else ["random0", "outside"]
        plans, plans_p, params, want_d, want_x = [], [], [], [], []
        for lab in labs:
            instr, values, gates, want = case(n, lab, K)
            plan = eng.compile(gates)
            sv = eng.statevector(plan, values)
            assert np.max(np.abs(sv - emulated(n, lab, K, R, False))) < tol_sv, (n, lab)
            assert np.max(np.abs(sv - want)) < tol_sv, (n, lab)
            cov.add(dc.plan_for(gates, K, R, False)[1])
            cov_drop.add(dc.plan_for(gates, K, R, True)[1])
            plans.append(plan), plans_p.append(eng.compile(gates, drop_final_phases=True)), params.append(values)
            want_d.append(float(np.dot(np.abs(want) ** 2, table))), want_x.append(oq.estimator_expectation(want, mixed))
            # |psi|^2 of the phase-dropped plan: sampling with identical uniforms (<= 1 boundary flip, to a CDF neighbour)
            shots = 2000
            u = np.random.default_rng(n + len(lab)).random(shots)
            got = eng.sample([plans_p[-1]], [values], shots, u.reshape(1, -1))[0]
            ref = oq.sample_indices(want, shots, uniforms=u)
            if single:  # complex64 probabilities differ at 1e-7 relative: flips to nearby states
                assert np.count_nonzero(np.abs(got - ref) > 64) <= shots // 100, (n, lab)
                continue
            probs = np.abs(emulated(n, lab, K, R, True)) ** 2
            bad = np.nonzero(got != ref)[0]
            assert len(bad) <= 1, (n, lab, len(bad))
            for i in bad:
                nz = np.flatnonzero(probs > 0)
                pos = np.searchsorted(nz, ref[i])
                assert got[i] in nz[max(0, pos - 1) : pos + 2], (n, lab, got[i], ref[i])
        for g, w in zip(eng.expectation(plans_p, params, ham_d), want_d):  # diagonal <H> through |psi|^2 (fused epilogue)
            assert rel_err(g, w) < tol_ev
        for g, w in zip(eng.expectation(plans, params, ham_x), want_x):  # Pauli sum with X / Y terms: the amplitudes route
            assert rel_err(g, w) < tol_ev
    print(f"\n{kind}: kept phases\n{cov.report()}\ndropped phases\n{cov_drop.report()}")
    assert cov.missing(False) == [] and cov_drop.missing(True) == []
    eng.close()


# ------------------------------------------------------------------------------------ b. start kinds
def test_zero_partial_and_prefix_starts():
    eng = make_engine()
    for n in (11, 13, 14):
        instr, values, gates, want = case(n, "zero", 11)
        plan = eng.compile(gates, from_zero_state=False)  # no product factor: the kernel synthesises |0...0> itself
        _, enc = dc.plan_for(gates, 11, 4, False, from_zero_state=False)
        assert np.all(enc[4] < 0)
        sv = eng.statevector(plan, values)
        assert np.max(np.abs(sv - emulated(n, "zero", 11, 4, False, False))) < 1e-13
        assert np.max(np.abs(sv - want)) < 1e-13
        instr, values, gates, want = case(n, "partial", 11)
        init = dc.plan_for(gates, 11, 4, False)[1][4][:n]
        assert 0 < np.count_nonzero(init >= 0) < n  # only some qubits fold into the product start
        assert np.max(np.abs(eng.statevector(eng.compile(gates), values) - want)) < 1e-13
    # cached prefix state: a parameter-free prefix over the general gate set, then a parameterised suffix
    n = 14
    diag, table, mixed = hamiltonians(n)
    ham_d = eng.hamiltonian(SparsePauliOp.from_list(diag))
    head = dc.random_circuit(n, 60, 5)
    head = oq.bind(head, dc.values_for(head, 6))
    instr = head + dc.random_circuit(n, 60, 7)
    gates = dc.gates_of(instr, n)
    for drop in (False, True):
        reuse = eng.compile_with_prefix_reuse(gates, drop_final_phases=drop)
        assert reuse.prefix is not None
        for seed in range(3):
            values = dc.values_for(instr, 50 + seed)
            want = oq.statevector(instr, n, values)
            if drop:
                assert rel_err(eng.expectation([reuse], [values], ham_d)[0], float(np.dot(np.abs(want) ** 2, table))) < 1e-10
            else:
                assert np.max(np.abs(eng.statevector(reuse, values) - want)) < 1e-13
    eng.close()


# ------------------------------------------------------------------------------------ c. tiles per CTA, batch composition
def _batch_rows(n, K):
    rows = []
    for i in range(32):
        lab = labels(n, K)[i % len(labels(n, K))]
        rows.append(lab)
    return rows


@pytest.mark.parametrize("tiles_log2", [0, 1, 2, 3])
def test_tiles_per_cta_and_batch_composition(monkeypatch, tiles_log2):
    monkeypatch.setenv("QB_TILES_LOG2", str(tiles_log2))
    eng = make_engine()
    n, K = 16, 11
    diag, table, _ = hamiltonians(n)
    ham = eng.hamiltonian(SparsePauliOp.from_list(diag))
    for lab in labels(n, K):
        _, values, gates, want = case(n, lab, K)
        assert np.max(np.abs(eng.statevector(eng.compile(gates), values) - want)) < 1e-13, lab
    rows = _batch_rows(n, K)
    for size in (1, 3, 32):
        sel = rows[:size] if size < 32 else rows
        plans = [eng.compile(case(n, lab, K)[2], drop_final_phases=True) for lab in sel]
        got = eng.expectation(plans, [case(n, lab, K)[1] for lab in sel], ham)
        for g, lab in zip(got, sel):
            assert rel_err(g, float(np.dot(np.abs(case(n, lab, K)[3]) ** 2, table))) < 1e-10, (size, lab)
    eng.close()


# ------------------------------------------------------------------------------------ d. launch switches
def _switch_outputs(eng, n=14, K=11):
    diag, table, mixed = hamiltonians(n)
    ham_d, ham_x = eng.hamiltonian(SparsePauliOp.from_list(diag)), eng.hamiltonian(SparsePauliOp.from_list(mixed))
    rows = _batch_rows(n, K)
    plans_p = [eng.compile(case(n, lab, K)[2], drop_final_phases=True) for lab in rows]
    plans = [eng.compile(case(n, lab, K)[2]) for lab in rows]
    params = [case(n, lab, K)[1] for lab in rows]
    out = [eng.expectation(plans_p, params, ham_d), eng.expectation(plans, params, ham_x)]
    rng = np.random.default_rng(3)
    for k in (1, 2, 3, 4):  # one circuit at 1-4 parameter points: the CUDA-graph path
        pts = [list(rng.uniform(-math.pi, math.pi, len(params[0]))) for _ in range(k)]
        out.append(eng.expectation([plans_p[0]] * k, pts, ham_d))
        out.append(eng.expectation([plans[0]] * k, pts, ham_x))
    out += [eng.statevector(plans[i], params[i]) for i in range(len(labels(n, K)))]
    return out


@pytest.fixture(scope="module")
def default_switch_outputs():
    eng = make_engine()
    out = _switch_outputs(eng)
    eng.close()
    return out


@pytest.mark.parametrize("name,value", [("QB_SWEEP_STREAMS", "1"), ("QB_SWEEP_GROUP", "2"), ("QB_PDL", "0"), ("QB_PDL", "2"), ("QB_GRAPHS", "0"),
                                        ("QB_ZERO_COPY", "0"), ("QB_L2_PREFETCH", "0")])
def test_launch_switches_are_bit_identical(monkeypatch, default_switch_outputs, name, value):
    """None of these switches changes per-amplitude arithmetic or a summation order."""
    monkeypatch.setenv(name, value)
    eng = make_engine()
    got = _switch_outputs(eng)
    eng.close()
    assert len(got) == len(default_switch_outputs)
    for a, b in zip(got, default_switch_outputs):
        assert np.array_equal(a, b)


# ------------------------------------------------------------------------------------ e. rank offsets of sharded segments
def _apply_reference(state, op, params):
    m = np.array(op.matrix(params))
    idx = np.arange(state.size)
    sel = ((idx >> op.target) & 1) == 0
    if op.control >= 0:
        sel &= ((idx >> op.control) & 1) == 1
    lo = idx[sel]
    hi = lo | (1 << op.target)
    x, y = state[lo].copy(), state[hi].copy()
    state[lo], state[hi] = m[0, 0] * x + m[0, 1] * y, m[1, 0] * x + m[1, 1] * y


@pytest.mark.parametrize("n_local,g", [(12, 2), (11, 3)])
def test_rank_offsets_of_sharded_segments(n_local, g):
    """Segments as the sharded backend builds them: dense targets on local qubits, controls and diagonal targets also on rank
    qubits (>= n_local), resolved per rank through index_offset = rank << n_local."""
    import torch

    eng = make_engine()
    n, world = n_local + g, 1 << g
    full_gates = dc.gates_of(dc.random_circuit(n, 160, n_local) + dc.outside_tile_circuit(n, 11, 1), n)
    ops = [op for op in full_gates.ops if op.kind == gl.DIAG or op.target < n_local]
    assert any(op.kind == gl.DIAG and op.target >= n_local for op in ops) and any(op.control >= n_local for op in ops)
    seg = gl.GateList(n_local, ops, full_gates.n_params, ())
    plan = eng.compile(seg, from_zero_state=False)
    values = list(np.random.default_rng(1).uniform(-math.pi, math.pi, full_gates.n_params))
    rng = np.random.default_rng(2)
    start = rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)
    start /= np.linalg.norm(start)
    for init_zero in (False, True):
        want = start.copy() if not init_zero else np.eye(1, 1 << n, dtype=complex)[0]
        for op in ops:
            _apply_reference(want, op, values)
        bufs = [torch.from_numpy(start[r << n_local : (r + 1) << n_local].copy()).cuda() for r in range(world)]
        torch.cuda.synchronize()
        for r in range(world):
            eng.apply_plan_device(plan, values, bufs[r].data_ptr(), init_zero, r << n_local)
        eng.synchronize()
        got = np.concatenate([b.cpu().numpy() for b in bufs])
        assert np.max(np.abs(got - want)) < 1e-13, init_zero
        if init_zero:
            assert not np.any(got[1 << n_local :])  # other ranks' slices stay exactly zero
    eng.close()


# ------------------------------------------------------------------------------------ sampler at the CDF edges
def _edge_uniforms(p):
    """0, nextafter(1, 0) and every CDF boundary c_k / c_last with its two float neighbours -> (uniforms, allowed index sets)."""
    nz = np.flatnonzero(p > 0)
    c = np.cumsum(p)
    c = c / c[-1]
    us, allowed = [0.0, np.nextafter(1.0, 0.0)], [{int(nz[0])}, {int(nz[-1])} | ({int(nz[-2])} if len(nz) > 1 else set())]
    for j, k in enumerate(nz[:-1]):
        for u in (np.nextafter(c[k], 0.0), c[k], np.nextafter(c[k], 1.0)):
            if 0.0 <= u < 1.0:
                us.append(float(u)), allowed.append({int(k), int(nz[j + 1])})
    return np.asarray(us), allowed


def _check_draws(got, p, n, us, allowed):
    c = np.cumsum(p)
    exact = np.searchsorted(c / c[-1], us, side="right")
    assert np.all(got < (1 << n)) and np.all(got >= 0)
    zero = got[p[got] == 0]
    assert zero.size == 0, f"{zero.size} draws of zero-probability indices, e.g. {zero[:5]}"
    for i, (gi, ok) in enumerate(zip(got, allowed)):
        assert gi in ok, (i, us[i], gi, exact[i], ok)
    assert exact[0] == got[0]


def _product_circuit(n, active, seed):
    rng = np.random.default_rng(seed)
    return [("ry", (q,), (float(rng.uniform(0.3, 2.8)),)) for q in active] + [("rz", (q,), (float(rng.uniform(-3, 3)),)) for q in active]


SAMPLER_STATES = {  # n -> qubits that leave |0>: zero-probability runs inside chunks, at chunk ends, top qubits in |0>
    4: [(0, 2), (1, 2)],
    8: [(0, 1, 5), (3, 6)],
    9: [(0, 8), (2, 3, 4, 5, 6, 7)],
    10: [(0, 1, 5, 9), (8,)],
    14: [tuple(range(8)), (0, 4, 8, 12, 13)],
}


@pytest.mark.parametrize("dtype", ["complex128", "complex64"])
def test_sampler_at_cdf_edges_through_circuits(dtype):
    eng = make_engine("c128" if dtype == "complex128" else "c64")
    for n, patterns in SAMPLER_STATES.items():
        for i, active in enumerate(patterns):
            instr = _product_circuit(n, active, n + i)
            plan = eng.compile(dc.gates_of(instr, n))
            sv = eng.statevector(plan, [])  # the state the sampler reads (same plan, same kernels)
            p = sv.real ** 2 + sv.imag ** 2
            us, allowed = _edge_uniforms(p)
            got = eng.sample([plan], [[]], len(us), us.reshape(1, -1))[0]
            _check_draws(got, p, n, us, allowed)
    eng.close()


@pytest.mark.parametrize("dtype", ["complex128", "complex64"])
def test_sampler_at_cdf_edges_on_device_states(dtype):
    """qb_sample_device (the sharded sampler's kernel) on states written directly: zero runs inside and at the end of chunks,
    whole zero chunks, an empty top half."""
    import torch

    eng = make_engine()
    np_dtype = np.complex128 if dtype == "complex128" else np.complex64
    for n in (9, 10, 14):
        rng = np.random.default_rng(n)
        size = 1 << n
        for pattern in range(3):
            psi = (rng.normal(size=size) + 1j * rng.normal(size=size)) * (rng.random(size) < 0.5)
            if pattern == 1:
                psi[size // 2 :] = 0  # top qubit |0>
                psi[480:512] = 0  # zero run at the end of the first chunk
            if pattern == 2:
                psi[: size // 4] = 0
                psi[np.arange(size) % 512 > 500] = 0
            psi = (psi / np.linalg.norm(psi)).astype(np_dtype)
            p = psi.real.astype(np.float64) ** 2 + psi.imag.astype(np.float64) ** 2
            us, allowed = _edge_uniforms(p)
            buf = torch.from_numpy(psi).cuda()
            torch.cuda.synchronize()
            got = eng.sample_device(dtype, n, buf.data_ptr(), us)
            _check_draws(got, p, n, us, allowed)
    eng.close()
