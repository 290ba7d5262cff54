"""One-GPU states of 26-34 qubits, across the 2^31 and 2^32 index boundaries, against the exact block-product references of
tests/wide_reference.py (pinned to the oracle by tests/test_wide_reference.py).

A single B200 holds 33 qubits in complex128 and 34 in complex64.  Several routes switch on only in that band: the 64-bit-index
sweep kernels (> 31 qubits), the on-the-fly diagonal <H> (table above a sixteenth of the workspace), the plain single-circuit
path (state above the CUDA-graph budget), the CVaR sort of more than INT_MAX pairs (31) over the full uint32 range (32), and
one-shot chunks of one to three states.  Every test checks the free device memory against the need written in it and skips
with the numbers when the state does not fit (the GPUs are shared); it uses one engine and closes it.  The module prints the
routes each width took at the end."""
import contextlib
import time

import numpy as np
import pytest

from queasars_b200 import expectation as ex
from queasars_b200.operators import SparsePauliOp
from tests import dispatch_coverage as dc
from tests import wide_reference as wr

pytestmark = pytest.mark.gpu

GiB = 1 << 30
MARGIN = 2 * GiB  # plans, partial sums, sampler chunks, CUDA context growth
TOL = {"complex128": 1e-10, "complex64": 1e-4}
WIDTHS = [("complex128", n) for n in (27, 29, 30, 31, 32, 33)] + [("complex64", n) for n in (31, 33, 34)]
IDS = [f"{'c128' if d == 'complex128' else 'c64'}-{n}q" for d, n in WIDTHS]
ROUTES: dict = {}


def amp_bytes(dtype):
    return 16 if dtype == "complex128" else 8


def rel_err(got, want):
    return abs(got - want) / max(1.0, abs(want))


def fit_or_skip(need: int, what: str):
    """An engine's workspace is 80 % of the device memory free when it is created: skip unless ``need`` bytes fit there."""
    import torch

    free, _ = torch.cuda.mem_get_info(0)
    usable = free // 10 * 8
    if need > usable:
        pytest.skip(f"{what}: needs {need / GiB:.1f} GiB, {usable / GiB:.1f} GiB usable of {free / GiB:.1f} GiB free on the device")


def note(dtype, n, **kv):
    ROUTES.setdefault((dtype, n), {}).update(kv)


@contextlib.contextmanager
def engine(dtype, n, **kw):
    from queasars_b200.engine import Engine

    t0 = time.perf_counter()
    eng = Engine(device=0, dtype=dtype, **kw)
    try:
        note(dtype, n, workspace=eng.workspace_bytes)
        yield eng
    finally:
        eng.close()
        r = ROUTES.setdefault((dtype, n), {})
        r["seconds"] = r.get("seconds", 0.0) + time.perf_counter() - t0


@pytest.fixture(scope="module", autouse=True)
def route_summary():
    yield
    print("\nwide-state routes (dtype, qubits: routes, workspace, seconds)")
    for (dtype, n), r in sorted(ROUTES.items(), key=lambda kv: (kv[0][0], kv[0][1])):
        rest = ", ".join(f"{k}={v}" for k, v in r.items() if k not in ("workspace", "seconds"))
        print(f"  {dtype:10s} {n:2d}q: {rest}; workspace {r.get('workspace', 0) / GiB:.1f} GiB; {r.get('seconds', 0.0):.1f} s")


def index_route(n):
    return "idx64" if n > 31 else "idx32"


def gates(lay):
    return dc.gates_of(lay.instr, lay.n)


# ------------------------------------------------------------------------------------ <H> through Engine.expectation
@pytest.mark.parametrize("dtype,n", WIDTHS, ids=IDS)
def test_expectation_pauli_sum_and_diagonal(dtype, n):
    state = amp_bytes(dtype) << n
    table = 8 << n
    fit_or_skip(state + (table if n <= 30 else 0) + MARGIN, f"{n}-qubit {dtype} state" + (" and its diagonal table" if n <= 30 else ""))
    lay = wr.dense_layout(n)
    tol = TOL[dtype]
    S = wr.ising_subset(n)
    _, _, dterms = wr.ising_on(n, S)
    with engine(dtype, n) as eng:
        g = gates(lay)
        # TFIM-like sum: X / Y on every high qubit, tile sweeps of x-mask groups and one group wider than a tile
        terms = wr.tfim_terms(n)
        got = eng.expectation([eng.compile(g)], [lay.values], eng.hamiltonian(SparsePauliOp.from_list(terms)))[0]
        assert rel_err(got, lay.pauli_sum(terms)) < tol
        # diagonal Ising on S: fused table epilogue against on-the-fly terms where the table fits, the default above
        want = lay.pauli_sum(dterms)
        plan = eng.compile(g, drop_final_phases=True)
        op = SparsePauliOp.from_list(dterms)
        if n <= 30:
            vals = {bt: eng.expectation([plan], [lay.values], eng.hamiltonian(op, build_table=bt))[0] for bt in (True, False)}
            for v in vals.values():
                assert rel_err(v, want) < tol
            assert abs(vals[True] - vals[False]) <= 1e-12 * max(1.0, abs(want))
            note(dtype, n, diag="table+on-the-fly")
        else:
            got = eng.expectation([plan], [lay.values], eng.hamiltonian(op))[0]
            assert rel_err(got, want) < tol
            note(dtype, n, diag="table" if table <= eng.workspace_bytes // 16 else "on-the-fly")
        budget = min(4 * GiB, eng.workspace_bytes // 8)
        note(dtype, n, sweeps=index_route(n), single="graph" if state <= budget // 4 else "plain")


@pytest.mark.parametrize("dtype,n", WIDTHS, ids=IDS)
def test_batch_of_three_in_chunks_of_two(dtype, n):
    """Three circuits with different sweep counts under a workspace for two states: chunks of 2 + 1, the first in a sorted
    device order that is not the caller's."""
    state = amp_bytes(dtype) << n
    fit_or_skip(2 * state + MARGIN, f"two resident {n}-qubit {dtype} states")
    lays = [wr.dense_layout(n, 1, 1), wr.dense_layout(n, 2, 5), wr.dense_layout(n, 3, 3)]
    terms = wr.tfim_terms(n)
    with engine(dtype, n, workspace_limit=2 * state + state // 2) as eng:
        plans = [eng.compile(gates(lay)) for lay in lays]
        assert plans[0].n_sweeps < plans[1].n_sweeps  # the first chunk runs entry 1 before entry 0
        got = eng.expectation(plans, [lay.values for lay in lays], eng.hamiltonian(SparsePauliOp.from_list(terms)))
        for g, lay in zip(got, lays):
            assert rel_err(g, lay.pauli_sum(terms)) < TOL[dtype]
        note(dtype, n, batch=f"2+1 sweeps {[p.n_sweeps for p in plans]}")


@pytest.mark.parametrize("dtype,n", [("complex128", 26), ("complex128", 27), ("complex64", 27), ("complex64", 28)])
def test_single_circuit_on_both_sides_of_the_graph_budget(dtype, n):
    state = amp_bytes(dtype) << n
    fit_or_skip(state + MARGIN, f"{n}-qubit {dtype} state")
    lay = wr.dense_layout(n)
    terms = wr.tfim_terms(n)
    with engine(dtype, n) as eng:
        plan = eng.compile(gates(lay))
        ham = eng.hamiltonian(SparsePauliOp.from_list(terms))
        a = eng.expectation([plan], [lay.values], ham)[0]
        b = eng.expectation([plan], [list(lay.values)], ham)[0]  # a replayed graph where it applies
        assert rel_err(a, lay.pauli_sum(terms)) < TOL[dtype]
        assert a == b
        budget = min(4 * GiB, eng.workspace_bytes // 8)
        note(dtype, n, single="graph" if state <= budget // 4 else "plain")


# ------------------------------------------------------------------------------------ sampling
def _sparse_allowed(support, p, us, eps):
    """Allowed draws of each uniform: the searchsorted entry, and its CDF neighbours where u lies within eps of a boundary."""
    c = np.cumsum(p)
    c = c / c[-1]
    j = np.searchsorted(c, us, side="right")
    out = []
    for u, jj in zip(us, j):
        ok = {int(support[min(jj, len(support) - 1)])}
        for b in np.flatnonzero(np.abs(c[:-1] - u) <= eps):
            ok |= {int(support[b]), int(support[b + 1])}
        out.append(ok)
    return out


@pytest.mark.parametrize("dtype,n", WIDTHS, ids=IDS)
def test_sampling_dense_and_sparse(dtype, n):
    state = amp_bytes(dtype) << n
    fit_or_skip(state + MARGIN, f"{n}-qubit {dtype} state")
    shots = 20000
    single = dtype == "complex64"
    with engine(dtype, n) as eng:
        # dense: index for index against the descent
        lay = wr.dense_layout(n)
        u = np.random.default_rng(n).random(shots)
        got = eng.sample([eng.compile(gates(lay), drop_final_phases=True)], [lay.values], shots, u.reshape(1, -1))[0]
        want = lay.sample(u)
        assert np.all((got >= 0) & (got < (1 << n)))
        diff = np.flatnonzero(got != want)
        if diff.size:
            assert np.all(lay.probabilities(got[diff]) > 0)
            lo, hi = np.minimum(got[diff], want[diff]), np.maximum(got[diff], want[diff])
            between = lay.mass_below(hi) - lay.mass_below(lo) - lay.probabilities(lo)  # mass strictly between the two draws
            # complex64: the CDF is as exact as float amplitudes; complex128: <= 1 boundary flip per 10^4 shots, to a neighbour
            assert np.max(between) < (1e-4 if single else 1e-10)
        if not single:
            assert diff.size <= shots // 10**4, f"{diff.size} of {shots} draws differ from the inverse CDF"
        # sparse: 64 indices on both sides of 2^31 / 2^32, exact against the sparse CDF, plus uniforms on its edges
        sp = wr.sparse_layout(n)
        support = wr.sparse_support(sp)
        p = sp.probabilities(support)
        c = np.cumsum(p) / np.sum(p)
        edges = [0.0, float(np.nextafter(1.0, 0.0))] + [float(x) for b in c[:-1] for x in (np.nextafter(b, 0.0), b, np.nextafter(b, 1.0))]
        us = np.concatenate([edges, np.random.default_rng(n + 1).random(shots)])
        got = eng.sample([eng.compile(gates(sp), drop_final_phases=True)], [sp.values], us.size, us.reshape(1, -1))[0]
        allowed = _sparse_allowed(support, p, us, 1e-6 if single else 1e-12)
        bad = [(i, float(us[i]), int(g)) for i, (g, ok) in enumerate(zip(got, allowed)) if int(g) not in ok]
        assert not bad, f"{len(bad)} sparse draws outside their allowed sets, e.g. {bad[:4]}"
        assert got[0] == support[0]
        note(dtype, n, sample=f"{diff.size} flips")


# ------------------------------------------------------------------------------------ observables
@pytest.mark.parametrize("dtype,n", WIDTHS, ids=IDS)
def test_observables(dtype, n):
    state = amp_bytes(dtype) << n
    fit_or_skip(state + MARGIN, f"{n}-qubit {dtype} state")
    lay = wr.dense_layout(n)
    obs = wr.observable_sets(n)
    with engine(dtype, n) as eng:
        handle = eng.observables([SparsePauliOp.from_list(o) for o in obs])
        got = eng.expectation_many([eng.compile(gates(lay))], [lay.values], handle)[0]
        for g, o in zip(got, obs):
            assert rel_err(g, lay.pauli_sum(o)) < TOL[dtype]


# ------------------------------------------------------------------------------------ exact CVaR
def cvar_expectation(alpha, n, dtype, workspace, sorted_built):
    """What ``qb_evaluate_cvar`` must do, from the byte counts of ``ensure_cvar_order`` and the check after it: 'sorted' /
    'unsorted' (runs), 'refused' (QB_ERR_MEMORY), 'too-wide' (QB_ERR_INVALID: 32-bit sorted order) or 'either' when the CUB
    sort storage, which only the device knows, decides."""
    size = 1 << n
    state = amp_bytes(dtype) << n
    if ex._close(alpha, 1):  # the energies, and the sorted order data when an earlier call built them
        return "unsorted" if (20 if sorted_built else 8) * size + state <= workspace else "refused"
    if n > 32:
        return "too-wide"
    kept = 20 * size
    build = kept + 4 * size + 12 * size  # + input indices + CUB's alternate key / value buffers
    if kept + state > workspace or build > workspace:
        return "refused"
    return "sorted" if build + build // 100 + (64 << 20) <= workspace else "either"


@pytest.mark.parametrize("dtype,n", WIDTHS, ids=IDS)
def test_exact_cvar(dtype, n):
    from queasars_b200 import _native

    state = amp_bytes(dtype) << n
    fit_or_skip(state + MARGIN, f"{n}-qubit {dtype} state")
    lay = wr.dense_layout(n)
    S = wr.ising_subset(n)
    z, c, dterms = wr.ising_on(n, S)
    routes, sorted_built = [], False
    with engine(dtype, n) as eng:
        plan = eng.compile(gates(lay), drop_final_phases=True)
        ham = eng.hamiltonian(SparsePauliOp.from_list(dterms), build_table=False)
        for alpha in (0.05, 0.3, 1.0):
            expect = cvar_expectation(alpha, n, dtype, eng.workspace_bytes, sorted_built)
            try:
                got = eng.cvar([plan], [lay.values], ham, alpha)[0]
            except _native.QbError as err:
                assert expect in ("refused", "either", "too-wide"), f"alpha={alpha}: expected {expect}, got {err}"
                assert err.code == (_native.QB_ERR_INVALID if expect == "too-wide" else _native.QB_ERR_MEMORY), str(err)
                routes.append(f"{alpha}:{'refused-idx32' if expect == 'too-wide' else 'refused'}")
                continue
            assert expect in ("sorted", "unsorted", "either"), f"alpha={alpha}: expected {expect}, got a value {got}"
            # knife edge: a stop bound moved by 1e-12 stands for the device's summation order
            cands = [lay.cvar(S, z, c, alpha, shift) for shift in (0.0, -1e-12, 1e-12)]
            err = min(abs(got - w) for w in cands) / max(1.0, abs(cands[0]))
            assert err <= TOL[dtype], f"alpha={alpha}: got {got!r}, reference {cands[0]!r} (rel {err:.2e})"
            sorted_built = sorted_built or expect != "unsorted"
            routes.append(f"{alpha}:{'sorted' if expect != 'unsorted' else 'unsorted'}")
    note(dtype, n, cvar=" ".join(routes))


def test_sorted_cvar_above_32_qubits_is_refused_before_any_allocation():
    """The sorted order stores basis indices as uint32: at 33 qubits they would wrap.  The refusal must not depend on the
    workspace being too small, so the workspace limit here is far above any device."""
    from queasars_b200 import _native

    n = 33
    lay = wr.dense_layout(n)
    S = wr.ising_subset(n)
    _, _, dterms = wr.ising_on(n, S)
    with engine("complex128", n, workspace_limit=1 << 42) as eng:
        plan = eng.compile(gates(lay), drop_final_phases=True)
        ham = eng.hamiltonian(SparsePauliOp.from_list(dterms), build_table=False)
        for alpha in (0.05, 0.9999):
            with pytest.raises(_native.QbError, match="32 bits") as err:
                eng.cvar([plan], [lay.values], ham, alpha)
            assert err.value.code == _native.QB_ERR_INVALID


# ------------------------------------------------------------------------------------ amplitudes at the index boundaries
def test_amplitudes_around_2_31_and_2_32_on_a_device_buffer():
    n, dtype = 32, "complex128"
    fit_or_skip((16 << n) + MARGIN, "a 64 GiB caller-owned 32-qubit state")
    lay = wr.dense_layout(n)
    tol = 1e-12 * lay.max_abs()
    rng = np.random.default_rng(32)
    starts = [0, (1 << 31) - 2048, (1 << 32) - 4096] + [int(s) for s in rng.integers(0, (1 << 32) - 4096, 8)]
    with engine(dtype, n) as eng:
        ptr = eng.device_alloc(16 << n)
        try:
            eng.apply_plan_device(eng.compile(gates(lay)), lay.values, ptr, True)
            for s in starts:
                out = eng.device_read(ptr, 16 * s, np.empty(4096, dtype=np.complex128))
                err = np.max(np.abs(out - lay.amplitudes(np.arange(s, s + 4096))))
                assert err <= tol, f"window at {s}: {err:.2e} > {tol:.2e}"
        finally:
            eng.device_free(ptr)
    note(dtype, n, device="apply_plan_device idx64")


def test_index_width_64_is_bit_identical_at_31_qubits():
    """The same 31-qubit program through the automatic 32-bit-index kernels and the forced 64-bit ones: same arithmetic."""
    import torch

    n, dtype = 31, "complex128"
    fit_or_skip(2 * (16 << n) + MARGIN, "two 32 GiB 31-qubit states")
    lay = wr.dense_layout(n)
    a = b = None
    try:
        with engine(dtype, n) as eng:
            plan = eng.compile(gates(lay))
            a = torch.empty(1 << n, dtype=torch.complex128, device="cuda:0")
            b = torch.empty(1 << n, dtype=torch.complex128, device="cuda:0")
            torch.cuda.synchronize()
            eng.apply_plan_device(plan, lay.values, a.data_ptr(), True)
            eng.set_index_width(64)
            eng.apply_plan_device(plan, lay.values, b.data_ptr(), True)
        step = 1 << 27
        for lo in range(0, 1 << n, step):
            assert torch.equal(a[lo : lo + step].view(torch.int64), b[lo : lo + step].view(torch.int64)), lo
        for s in ((1 << 30) - 2048, (1 << 31) - 4096):
            got = a[s : s + 4096].cpu().numpy()
            assert np.max(np.abs(got - lay.amplitudes(np.arange(s, s + 4096)))) <= 1e-12 * lay.max_abs()
    finally:
        del a, b
        torch.cuda.empty_cache()
    note(dtype, n, device="idx32 == idx64 bitwise")
