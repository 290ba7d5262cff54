"""The block-product reference of tests/wide_reference.py against the full NumPy oracle at 12-16 qubits, and the planner's reach on
the 31-34-qubit circuits the GPU tests run (tests/test_gpu_wide_states.py).  No GPU needed.

The reference is what the wide GPU tests trust, so it is pinned here on layouts of the same kind (interleaved blocks, X / Y and
controls on the high qubits, ties in the energies): amplitudes, Pauli sums, observables, inverse-CDF draws and exact CVaR with
its stop entry."""
import math

import numpy as np
import pytest

from oracle import qiskit_semantics as oq
from queasars_b200 import expectation as ex
from queasars_b200 import gate_list as gl
from queasars_b200.schedule import K_EXT
from tests import dispatch_coverage as dc
from tests import wide_reference as wr

SMALL = [(12, 4), (14, 5), (16, 6)]  # (n, block size): three or four interleaved blocks


def oracle_state(lay):
    return oq.statevector(lay.instr, lay.n, lay.values)


@pytest.fixture(scope="module", params=SMALL, ids=lambda p: f"{p[0]}q")
def small(request):
    n, bm = request.param
    lay = wr.dense_layout(n, 1, 3, bm)
    assert len(lay.blocks) >= 3 and all(len(b.qubits) <= bm for b in lay.blocks)
    return lay, oracle_state(lay)


def test_amplitudes(small):
    lay, psi = small
    got = lay.amplitudes(np.arange(psi.size))
    assert np.max(np.abs(got - psi)) < 1e-14
    assert lay.max_abs() == pytest.approx(np.max(np.abs(psi)), rel=1e-12)


def test_pauli_sums_and_observables(small):
    lay, psi = small
    n = lay.n
    rng = np.random.default_rng(n)
    mixed = [("".join(rng.choice(list("IXYZ"), size=n, p=[0.5, 0.2, 0.15, 0.15])), complex(rng.normal(), rng.normal())) for _ in range(24)]
    for terms in [wr.tfim_terms(n), mixed] + wr.observable_sets(n):
        assert lay.pauli_sum(terms) == pytest.approx(oq.estimator_expectation(psi, terms), rel=1e-12, abs=1e-13)
    for lab, _ in mixed:
        assert abs(lay.pauli(lab) - oq.pauli_expectation(psi, lab)) < 1e-13


def test_inverse_cdf_draws(small):
    lay, psi = small
    p = psi.real**2 + psi.imag**2
    cdf = np.cumsum(p)
    u = np.concatenate([[0.0, np.nextafter(1.0, 0.0)], np.random.default_rng(3).random(3000)])
    want = oq.sample_indices(psi, 0, uniforms=u)
    assert np.array_equal(lay.sample(u), want)
    for x in u[:40]:  # the scalar descent (the one the CVaR stop entry uses) with searchsorted's side='right'
        assert lay.descend(float(x) * cdf[-1], side="right")[0] == cdf.searchsorted(x * cdf[-1], side="right")
    # side='left' with the running mass before the entry and the entry's own mass
    for x in u[2:40]:
        k, before, pk = lay.descend(float(x))
        assert k == int(np.searchsorted(cdf, x, side="left"))
        assert before == pytest.approx(cdf[k] - p[k], abs=1e-14) and pk == pytest.approx(p[k], rel=1e-12, abs=1e-16)
        assert lay.measure_below(k) == pytest.approx(before, abs=1e-14)
    ks = np.random.default_rng(4).integers(0, psi.size, 200)
    assert np.max(np.abs(lay.mass_below(ks) - (cdf[ks] - p[ks]))) < 1e-14


def test_sparse_layout_support_and_draws():
    n = 14
    lay = wr.sparse_layout(n)
    psi = oracle_state(lay)
    p = psi.real**2 + psi.imag**2
    support = wr.sparse_support(lay)
    assert support.size == 64 and set(np.flatnonzero(p)) <= set(support.tolist())
    assert np.max(np.abs(lay.amplitudes(support) - psi[support])) < 1e-15
    u = np.concatenate([[0.0, np.nextafter(1.0, 0.0)], np.random.default_rng(5).random(500)])
    assert np.array_equal(lay.sample(u), oq.sample_indices(psi, 0, uniforms=u))
    c = np.cumsum(p[support])
    for j, cj in enumerate(c[:-1] / c[-1]):  # on a CDF boundary: one of the two entries that meet there
        for x in (np.nextafter(cj, 0.0), cj, np.nextafter(cj, 1.0)):
            assert lay.sample([x])[0] in (support[j], support[j + 1])
    assert wr.sparse_active(34) == [0, 1, 30, 31, 32, 33]


def _oracle_stop(p, table, alpha):
    """Basis index at which lower_tail_expectation_arrays stops."""
    order = np.arange(p.size) if ex._close(alpha, 1) else np.argsort(table, kind="stable")
    cum = np.cumsum(p[order])
    return int(order[np.nonzero(cum >= alpha - (ex._ATOL + ex._RTOL * alpha))[0][0]])


ALPHAS = (0.05, 0.3, 0.5, 0.77, 0.9999, 1 - 5e-6, 1.0)


def _hamiltonians(n):
    S = wr.ising_subset(n)
    z, c, _ = wr.ising_on(n, S)
    hq = wr.high_qubits(n)
    sym = sorted({0, 5, 10, 11, *hq[:3]})
    return [
        ("ising", S, z, c),
        # sum of Z with one coefficient: binomially large tie groups that span many S-patterns
        ("ties", sym, [1 << q for q in sym], [1.0] * len(sym)),
        # two energies of about half the mass each: every alpha < 1/2 stops inside one tie group of 2^(n-1) entries
        ("halves", sorted([3, hq[-1]]), [(1 << 3) | (1 << hq[-1])], [1.0]),
    ]


def test_cvar_value_and_stop_entry(small):
    lay, psi = small
    n = lay.n
    p = psi.real**2 + psi.imag**2
    for name, S, z, c in _hamiltonians(n):
        table = oq.diagonal_table(n, list(zip(z, c)))
        assert np.array_equal(np.unique(table), np.unique(wr.Layout.pattern_energies(S, z, c)))
        masses = lay.pattern_masses(S)
        assert math.fsum(masses) == pytest.approx(1.0, abs=1e-13)
        for alpha in ALPHAS:
            got, k = lay.cvar_stop(S, z, c, alpha)
            want = ex.lower_tail_expectation_arrays(p, table, alpha)
            assert abs(got - want) <= 1e-12 * max(1.0, abs(want)), (name, alpha, got, want)
            assert k == _oracle_stop(p, table, alpha), (name, alpha)
            if name == "halves" and alpha < 0.45:
                assert np.count_nonzero(table == table[k]) == 1 << (n - 1)  # the stop entry is inside a large tie group


def test_cvar_shifted_stop_is_visible(small):
    """A stop entry one place early in its tie group is wrong by about the isclose width: the comparisons above detect it."""
    lay, psi = small
    n = lay.n
    p = psi.real**2 + psi.imag**2
    _, S, z, c = _hamiltonians(n)[2]
    table = oq.diagonal_table(n, list(zip(z, c)))
    alpha = 0.3
    order = np.argsort(table, kind="stable")
    cum = np.cumsum(p[order])
    s = int(np.nonzero(cum >= alpha - (ex._ATOL + ex._RTOL * alpha))[0][0])
    early = (float(np.dot(p[order[:s - 1]], table[order[:s - 1]])) + p[order[s - 1]] * table[order[s - 1]]) / alpha
    assert abs(early - lay.cvar(S, z, c, alpha)) > 1e-7


# ------------------------------------------------------------------------------------------------ planner reach
CONFIGS = [(11, 4), (12, 4), (11, 3)]
WIDE = (31, 32, 33, 34)


@pytest.mark.parametrize("drop", [False, True])
@pytest.mark.parametrize("tile_bits,reg_bits", CONFIGS)
def test_wide_plans_reach_the_high_index_bits(tile_bits, reg_bits, drop):
    """The plans of the wide GPU tests hold qubits >= 31 in sweep tiles, apply controls and diagonals on 31-33 from outside the
    tile, and fold every qubit into the product-state start; a planner change that moves them off these paths fails here."""
    ext_ctrl, ext_diag = set(), set()
    for n in WIDE:
        lay = wr.dense_layout(n)
        sweeps, passes, pass_ops, angles, init = dc.plan_for(dc.gates_of(lay.instr, n), tile_bits, reg_bits, drop)[1]
        tiles = [set(s["tile_qubits"][:tile_bits].tolist()) for s in sweeps]
        if n > 31:
            assert any(max(t) >= 31 for t in tiles), n
        assert max(max(t) for t in tiles) == n - 1
        assert int(np.count_nonzero(init >= 0)) == n == len(init)
        for po, _ in dc.plan_records((sweeps, passes, pass_ops, angles, init)):
            if int(po["ctrl_kind"]) == K_EXT:
                ext_ctrl.add(int(po["ctrl_qubit"]))
            if int(po["kind"]) == gl.DIAG and int(po["tgt_kind"]) == K_EXT:
                ext_diag.add(int(po["tgt_qubit"]))
    assert {31, 32, 33} <= ext_ctrl
    assert {31, 32} <= ext_diag


def test_wide_layouts_interleave_blocks():
    for n in WIDE + (27, 29, 30):
        lay = wr.dense_layout(n)
        assert all(len(b.qubits) <= wr.BLOCK_MAX for b in lay.blocks)
        for b in lay.blocks:  # every block holds low qubits, one of the tile-boundary qubits and high ones
            assert min(b.qubits) < 3 and set(b.qubits) & {10, 11, 12} and set(b.qubits) & set(wr.high_qubits(n))
        owner = [lay.block_of[q[0]][0] for _, q, _ in lay.instr]
        assert sum(a != b for a, b in zip(owner, owner[1:])) > len(owner) // 3  # blocks alternate in time
