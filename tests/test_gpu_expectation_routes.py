"""Every route of the Pauli-sum expectation kernels on the GPU, against a plain reduction of the same amplitudes: the fused
diagonal epilogue with and without the state store, the on-the-fly diagonal group (staged / unstaged terms), tile sweeps
(register and shared-memory partners, general groups, several sweeps and groups), generic groups (staged / unstaged), an
unusable tile plan, operators without terms, and the device-pointer route of sharded states with rank offsets.
tests/test_expectation_routes.py checks on the CPU that the operators used here reach every route.

Reference and tolerance.  The amplitudes are read back with ``Engine.statevector`` from the same plan and parameters, so the
comparison isolates the reduction.  Every term's value is reduced on its own in float64 (``expectation_routes.reference``) and
the terms are summed exactly with ``math.fsum``.  The kernels also accumulate in double, complex64 amplitudes included (a
product of two floats is exact in double), so the difference is rounding of double-precision sums alone.  With u = 2^-53, a
group's W(k) = sum_t ±w_t over T terms (or a table entry over the diagonal terms) is off by at most T·u·sum|w|, and the sum
over amplitudes, the per-thread accumulation over the groups of a tile sweep (8 amplitudes per group), the CTA reduction, the
partials reduction and the accumulation over launches add at most (8·G + 256)·u·sum|c|·|psi|^2 for G groups, because
sum_k |psi_k||psi_{k^x}| <= |psi|^2.  The reference's own error (pairwise sums or n butterfly levels per term) is below
64·u·|c_t| per term.  So |GPU - reference| <= (2·(T_max + 8·G) + 512)·u·sum|c_t|·max(1, |psi|^2): about 1e-13·sum|c_t| for
the small operators and 1.4e-12·sum|c_t| for 6001 diagonal terms (``expectation_routes.tolerance``), in both dtypes.  A
kernel that accumulated in float, or lost one tile's partial, misses it by orders of magnitude.  The oracle comparison of the
parity tests stays as well (1e-10 relative in complex128, 1e-4 in complex64, against ``oracle.qiskit_semantics``).

From 20 qubits on, the tiles per sweep CTA follow the batch size, and a state simulated alone can differ in its last bit from
the same state in a larger batch (DESIGN.md §4.8).  So at 20 qubits the tight comparison is made on batches of one and
multi-plan batches are compared with the oracle; bit-identity across batch compositions is checked at 16 qubits."""
import functools
import math

import numpy as np
import pytest

from oracle import evqe_genome as og
from oracle import qiskit_semantics as oq
from queasars_b200 import gate_list as gl
from tests import dispatch_coverage as dc
from tests import expectation_routes as er
from tests.test_frontend_planner import build_circuit

pytestmark = pytest.mark.gpu

BUILDS = [("c128", (1, 4, 10, 11, 12, 13, 16, 20)), ("c64", (1, 4, 10, 11, 12, 13, 16, 20)), ("tile12", (4, 11, 12))]
CASES = [(kind, n) for kind, widths in BUILDS for n in widths]


def make_engine(kind="c128"):
    from queasars_b200.engine import Engine

    return Engine(device=0, **{"c64": {"dtype": "complex64"}, "tile12": {"tile_bits": 12}}.get(kind, {}))


def circuits(n):
    """(label, instructions, gate list, parameter points): an EVQE individual and a random circuit over the whole gate set."""
    genome, values = og.random_individual(n, 3, True, 40 + n)
    out = [("evqe", og.individual_circuit(genome, values), list(values))]
    if n >= 2:
        instr = dc.random_circuit(n, 80, 7 * n)
        out.append(("random", instr, dc.values_for(instr, n)))
    res = []
    for label, instr, values in out:
        rng = np.random.default_rng(len(values) + n)
        points = [values] + [list(rng.uniform(-math.pi, math.pi, len(values))) for _ in range(3)]
        res.append((label, instr, gl.from_circuit(build_circuit(instr, n)), points))
    return res


@functools.lru_cache(maxsize=None)
def family(n, many_terms=None):
    return er.operator_family(n, many_terms=many_terms)


@functools.lru_cache(maxsize=None)
def oracle_state(n, ci):
    _, instr, _, points = circuits(n)[ci]
    return oq.statevector(instr, n, points[0])


@functools.lru_cache(maxsize=None)
def oracle_value(n, label, ci):
    """Reference value of the family operator ``label`` on the oracle's state of circuit ``ci`` (shared by the builds)."""
    op = dict((lab, o) for lab, o, _ in family(n))[label]
    return er.reference(oracle_state(n, ci), *op.masks())


def build_flag(eng, op, flag):
    """The build_table that ``Engine.hamiltonian(op, flag)`` uses."""
    if flag is not None:
        return flag
    n_diag = int(np.count_nonzero(op.masks()[0] == 0))
    return er.default_build_table(n_diag, op.num_qubits, eng.tile_bits, eng.workspace_bytes)


def upload(eng, op, flag):
    """-> (Hamiltonian handle, restated layout); the table builder's launches must match the restated chunk count."""
    before = eng.launch_count
    ham = eng.hamiltonian(op, build_table=flag)
    lay = er.layout_of(op, build_flag(eng, op, flag))
    assert eng.launch_count - before == lay.table_chunks
    return ham, lay


def oracle_close(got, want, op, single):
    scale = float(np.sum(np.abs(op.coeffs)))
    tol = (1e-4 * max(1.0, abs(want)) + 1e-5 * scale) if single else (1e-10 * max(1.0, abs(want)) + 1e-12 * scale)
    return abs(got - want) <= tol


def check(got, psi, op, lay, what, want=None):
    """|got - reference| within the double-precision reduction bound."""
    want = er.reference(psi, *op.masks()) if want is None else want
    norm2 = float(np.sum(psi.real ** 2 + psi.imag ** 2))
    tol = er.tolerance(lay, norm2)
    assert abs(got - want) <= tol, (what, got, want, abs(got - want), tol)
    return want


# ------------------------------------------------------------------------------------ a. every batched route, every entry point
@pytest.mark.parametrize("kind,n", CASES)
def test_every_route_through_every_entry_point(kind, n):
    eng = make_engine(kind)
    single = eng.dtype == "complex64"
    n_eff = max(n, eng.tile_bits)
    circs = circuits(n)
    plans = [eng.compile(gates) for _, _, gates, _ in circs]
    states = [[eng.statevector(p, pt) for pt in points] for p, (_, _, _, points) in zip(plans, circs)]
    seen = set()
    for label, op, flag in family(n):
        ham, lay = upload(eng, op, flag)
        routes, launches = er.batch_routes(lay, n_eff)
        seen |= er.features(lay, routes)
        what = (kind, n, label)
        refs = {}

        def ref(ci, j):  # reference of parameter point j of circuit ci (each computed once)
            if (ci, j) not in refs:
                refs[ci, j] = er.reference(states[ci][j], *op.masks())
            return refs[ci, j]

        for ci, (plan, (_, _, _, points)) in enumerate(zip(plans, circs)):
            # resident batch of one plan (the bench's path): the launch count binds the restated routes to the native planner
            rb = eng.resident_batch([plan], ham)
            rb.set_params([points[0]])
            rb.run()
            value = rb.read()[0]
            st = rb.stats()
            assert st["kernel_launches"] - 1 - st["sweep_launches"] == launches, (what, routes)
            rb.close()
            check(value, states[ci][0], op, lay, what + ("resident",), ref(ci, 0))
            assert oracle_close(value, oracle_value(n, label, ci), op, single), what
            if label == "empty":
                assert value == 0.0
            if label == "identity":
                assert abs(value - 1.25 * float(np.sum(np.abs(states[ci][0]) ** 2))) <= er.tolerance(lay, 1.0)
            # one circuit at 1-4 parameter points: the cached CUDA graph, bit-identical to the resident batch for the same point
            for k in (1, 2, 3, 4):
                got = eng.expectation([plan] * k, [list(p) for p in points[:k]], ham)
                assert got[0] == value, (what, k)
                for j in range(1, k if n_eff < 20 else min(k, 2)):  # (20 q: the reference of one more point suffices)
                    check(got[j], states[ci][j], op, lay, what + ("graph", k, j), ref(ci, j))
            assert eng.expectation([plan], [list(points[0])], ham)[0] == value  # repeated call
        # >= 5 plans in one call, and the same list through submit / collect (the pipelined path's native calls)
        batch_plans = [plans[i % len(plans)] for i in range(6)]
        slots = [(i % len(plans), (i // len(plans)) % 4) for i in range(6)]  # (circuit, parameter point) of every entry
        batch_params = [list(circs[ci][3][j]) for ci, j in slots]
        got = eng.expectation(batch_plans, batch_params, ham)
        eng.expectation_submit(batch_plans, batch_params, ham)
        piped = eng.expectation_collect(len(batch_plans))
        assert np.array_equal(got, piped), what
        for i, (g, (ci, j)) in enumerate(zip(got, slots)):
            if n_eff < 20:
                check(g, states[ci][j], op, lay, what + ("batch", i), ref(ci, j))
                assert g == eng.expectation([plans[ci]], [list(circs[ci][3][j])], ham)[0], (what, i)  # batch composition
            elif j == 0:
                assert oracle_close(g, oracle_value(n, label, ci), op, single), (what, i)
        if label == "empty":
            assert not np.any(got)
    print(f"\n{kind} n={n}: {sorted(seen)}")
    eng.close()


# ------------------------------------------------------------------------------------ b. launch switches of the graph path
@pytest.mark.parametrize("kind", ["c128", "c64"])
def test_graph_path_without_zero_copy_is_bit_identical(monkeypatch, kind):
    out = {}
    for zero_copy in ("1", "0"):
        monkeypatch.setenv("QB_ZERO_COPY", zero_copy)
        eng = make_engine(kind)
        vals = []
        for n in (4, 12, 16):
            circs = circuits(n)
            plans = [eng.compile(gates) for _, _, gates, _ in circs]
            for label, op, flag in family(n, many_terms=False):
                ham, lay = upload(eng, op, flag)
                for plan, (_, _, _, points) in zip(plans, circs):
                    for k in (1, 2, 3, 4):
                        got = eng.expectation([plan] * k, [list(p) for p in points[:k]], ham)
                        if zero_copy == "0" and k == 1:
                            check(got[0], eng.statevector(plan, points[0]), op, lay, (kind, n, label))
                        vals.append(got)
        out[zero_copy] = vals
        eng.close()
    assert len(out["1"]) == len(out["0"])
    for a, b in zip(out["1"], out["0"]):
        assert np.array_equal(a, b)


# ------------------------------------------------------------------------------------ c. the pipelined submission
@pytest.mark.parametrize("n", [12, 13, 16])
def test_pipelined_submission_on_every_route(n):
    eng = make_engine()
    eng._pipeline = True  # (off by default when the C marshalling helper is present)
    plans, params, states = [], [], []
    for seed in range(16):
        genome, values = og.random_individual(n, 6, True, 500 + seed)
        plans.append(eng.compile(gl.from_circuit(build_circuit(og.individual_circuit(genome, values), n))))
        params.append([float(v) for v in values])
        states.append(eng.statevector(plans[-1], values) if seed % 5 == 0 else None)
    assert eng._pipeline_split(plans, params) is not None and eng._pipeline_split(plans, [np.asarray(p) for p in params]) is None
    for label, op, flag in family(n):
        ham, lay = upload(eng, op, flag)
        piped = eng.expectation(plans, params, ham)
        whole = eng.expectation(plans, [np.asarray(p) for p in params], ham)  # arrays: submitted in one piece
        assert np.array_equal(piped, whole), label
        for i, psi in enumerate(states):
            if psi is not None:
                check(piped[i], psi, op, lay, (n, label, i))
    eng.close()


# ------------------------------------------------------------------------------------ d. the device-pointer route (sharded states)
@pytest.mark.parametrize("dtype", ["complex128", "complex64"])
def test_device_route_on_slices_with_rank_offsets(dtype):
    """A random state of 2^n amplitudes written into 2^g buffers of 2^n_local; qb_expectation_device per slice at index_offset =
    r << n_local, summed, against the full-state reference.  Also the table route on the whole state, and an X on a rank bit."""
    import torch

    from queasars_b200 import _native

    eng = make_engine()
    np_dtype = np.complex128 if dtype == "complex128" else np.complex64
    seen = set()
    for n_local in (9, 10, 11, 12, 14):
        for g in (1, 2, 3):
            n = n_local + g
            rng = np.random.default_rng(31 * n_local + g)
            psi = rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)
            psi = (psi / np.linalg.norm(psi)).astype(np_dtype)
            exact = psi.astype(np.complex128)
            bufs = [torch.from_numpy(psi[r << n_local : (r + 1) << n_local].copy()).cuda() for r in range(1 << g)]
            whole = torch.from_numpy(psi.copy()).cuda()
            torch.cuda.synchronize()
            for label, op, flag in er.device_family(n, n_local):
                ham, lay = upload(eng, op, bool(flag))
                before, predicted, vals = eng.launch_count, 0, []
                for r in range(1 << g):
                    routes, launches = er.device_routes(lay, n_local, r << n_local)
                    seen |= er.features(lay, routes, device_n_local=n_local)
                    predicted += launches
                    vals.append(eng.expectation_device(ham, dtype, n_local, bufs[r].data_ptr(), r << n_local))
                assert eng.launch_count - before == predicted, (n_local, g, label)
                check(sum(vals), exact, op, lay, (dtype, n_local, g, label))
                if label == "empty":
                    assert vals == [0.0] * len(vals)
                if flag and n >= er.TABLE_TILE_BITS:  # V1: the table of the full width, read by the table kernel
                    routes, launches = er.device_routes(lay, n, 0)
                    assert routes[0][0] == "V1"
                    seen.add("V1")
                    before = eng.launch_count
                    check(eng.expectation_device(ham, dtype, n, whole.data_ptr(), 0), exact, op, lay, (dtype, n, label, "V1"))
                    assert eng.launch_count - before == launches
            bad = er._op(n, [1 << n_local, 1], [0, 1 << (n - 1)], [1.0, 0.5])  # an X on the lowest rank bit
            ham = eng.hamiltonian(bad)
            with pytest.raises(_native.QbError) as err:
                eng.expectation_device(ham, dtype, n_local, bufs[0].data_ptr(), 0)
            assert err.value.code == _native.QB_ERR_INVALID
            del bufs, whole
    assert {"V1", "V2", "V3", "V4", "V5", "T1"} <= seen, sorted(seen)
    eng.close()
