"""Reach of the Pauli-sum expectation routes on the CPU: the operators of tests/expectation_routes.py must reach every route
class, every register partner distance S and every shared-memory staging boundary at the widths and builds that
tests/test_gpu_expectation_routes.py runs, so that those GPU tests cannot silently stop exercising a kernel branch when the
planner changes.  The route emulator then reproduces the oracle on random states, which checks the restated planner (tile
qubits, xloc, groups, table chunks) against the operator it encodes."""
import numpy as np
import pytest

from oracle import qiskit_semantics as oq
from tests import expectation_routes as er

WORKSPACE = 8 << 30  # (any workspace of a B200 builds the tables of these widths)

# (tile bits of the engine, widths): the GPU file's builds
BATCH_BUILDS = [(11, (1, 4, 10, 11, 12, 13, 16, 20)), (12, (4, 11, 12))]
DEVICE_SPLITS = [(n_local, g) for n_local in (9, 10, 11, 12, 14) for g in (1, 2, 3)]

BATCH_CLASSES = {"D1", "D2", "D3", "D4", "D5", "T1", "T2", "T3", "G1", "G2", "E0"}
BATCH_FEATURES = {"T1.S1", "T1.S2", "T1.S4", "T3.evenY", "T3.oddY", "T3.complex", "T4.sweeps", "T4.groups", "T5",
                  "stage.2000.diag", "stage.2001.diag", "stage.2000.group", "stage.2001.group", "table.chunks1", "table.chunks2", "table.chunks3"}
DEVICE_CLASSES = {"V1", "V2", "V3", "V5", "E0"}
DEVICE_FEATURES = {"V4", "T1", "T3.oddY", "T3.complex"}


def build_table_of(op, flag, tile_bits):
    if flag is not None:
        return flag
    n_diag = int(np.count_nonzero(op.masks()[0] == 0))
    return er.default_build_table(n_diag, op.num_qubits, tile_bits, WORKSPACE)


def batch_cases():
    """(tile bits, n, label, layout, routes, launches) of every operator the GPU file evaluates through the batched route."""
    for tile_bits, widths in BATCH_BUILDS:
        for n in widths:
            for label, op, flag in er.operator_family(n):
                lay = er.layout_of(op, build_table_of(op, flag, tile_bits))
                routes, launches = er.batch_routes(lay, max(n, tile_bits))
                yield tile_bits, n, label, lay, routes, launches


def device_cases():
    for n_local, g in DEVICE_SPLITS:
        n = n_local + g
        for label, op, flag in er.device_family(n, n_local):
            lay = er.layout_of(op, bool(flag))
            for r in range(1 << g):
                yield n_local, g, r, label, lay, er.device_routes(lay, n_local, r << n_local)
            if flag and er.TABLE_TILE_BITS <= n:  # the whole state as one slice: the table route
                yield n, 0, 0, label, lay, er.device_routes(lay, n, 0)


def test_family_reaches_every_batched_route():
    seen, by_build = set(), {}
    for tile_bits, n, label, lay, routes, launches in batch_cases():
        f = er.features(lay, routes)
        seen |= f
        by_build.setdefault(tile_bits, set()).update(f)
        assert launches == 2 * len({si for _, _, si in routes if si is not None}) + sum(
            {"D1": 1, "D2": 1, "E0": 1}.get(c, 0 if si is not None else 2) for c, _, si in routes)
    print("\nbatched route classes reached:", sorted(seen))
    assert BATCH_CLASSES | BATCH_FEATURES <= seen, sorted((BATCH_CLASSES | BATCH_FEATURES) - seen)
    assert {"T5", "D5"} <= by_build[12] and not {"T5", "D5"} & by_build[11]  # only a 12-bit-tile engine below 12 qubits


def test_family_reaches_every_device_route():
    seen = set()
    for n_local, g, r, label, lay, (routes, launches) in device_cases():
        seen |= er.features(lay, routes, device_n_local=n_local)
    print("\ndevice route classes reached:", sorted(seen))
    assert DEVICE_CLASSES | DEVICE_FEATURES <= seen, sorted((DEVICE_CLASSES | DEVICE_FEATURES) - seen)


def test_flips_on_rank_bits_are_refused():
    op = er._op(12, [1 << 11, 1], [0, 0], [1.0, 1.0])
    lay = er.layout_of(op, False)
    for n_local in (9, 11):
        with pytest.raises(er.RouteError):
            er.device_routes(lay, n_local, 0)


def test_restated_planner_matches_known_plans():
    """Hand-checked plans: a 16-qubit TFIM puts X_0..X_10 into one sweep on qubits 0..10 and X_11..X_15 into a second one on
    qubits 0..5 and 11..15; a lone X_8 / X_9 / X_10 lands on tile-local bit 8 / 9 / 10 (register partners, S = 1 / 2 / 4)."""
    lay = er.layout_of(er._op(16, *er._tfim(16, np.random.default_rng(0))), False)
    assert [sw.tile_qubits for sw in lay.sweeps] == [list(range(11)), list(range(6)) + list(range(11, 16))]
    assert [len(sw.groups) for sw in lay.sweeps] == [11, 5] and lay.generic == []
    for q, s in ((8, 1), (9, 2), (10, 4)):
        lay = er.layout_of(er._op(13, [1 << q], [0], [1.0]), None)
        routes, launches = er.batch_routes(lay, 13)
        assert routes == [("T1", 0, 0)] and launches == 2 and lay.groups[0].xloc >> 8 == s
    wide = er.layout_of(er._op(12, [0xFF << 4, 1], [0, 0], [1.0, 1.0]), None)
    assert wide.generic == [0] and er.batch_routes(wide, 12)[0] == [("T2", 1, 0), ("G1", 0, None)]
    assert er.batch_routes(er.layout_of(er._op(5, [], [], []), None), 11) == ([("E0", None, None)], 1)


def _random_state(n, seed):
    rng = np.random.default_rng(seed)
    psi = rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)
    return psi / np.linalg.norm(psi)


@pytest.mark.parametrize("tile_bits,n", [(11, 4), (11, 11), (11, 12), (11, 13), (12, 11)])
def test_emulator_reproduces_the_oracle(tile_bits, n):
    n_eff = max(n, tile_bits)
    psi = _random_state(n, 7 * n + tile_bits)
    padded = np.zeros(1 << n_eff, dtype=complex)
    padded[: psi.size] = psi
    for label, op, flag in er.operator_family(n):
        lay = er.layout_of(op, build_table_of(op, flag, tile_bits))
        routes, _ = er.batch_routes(lay, n_eff)
        want = oq.estimator_expectation(psi, op.to_list()) if op.size else 0.0
        got = er.emulate(lay, routes, padded, n_eff)
        assert abs(got - want) <= 1e-13 * max(1.0, float(np.sum(np.abs(op.coeffs)))), (label, got, want)
        ref = er.reference(psi, *op.masks())
        assert abs(ref - want) <= 1e-13 * max(1.0, float(np.sum(np.abs(op.coeffs)))), (label, ref, want)


@pytest.mark.parametrize("n_local,g", [(9, 2), (11, 1), (12, 2)])
def test_emulator_reproduces_the_oracle_on_slices(n_local, g):
    n = n_local + g
    psi = _random_state(n, n_local)
    for label, op, flag in er.device_family(n, n_local):
        lay = er.layout_of(op, bool(flag))
        want = oq.estimator_expectation(psi, op.to_list()) if op.size else 0.0
        got = sum(er.emulate(lay, er.device_routes(lay, n_local, r << n_local)[0], psi[r << n_local : (r + 1) << n_local], n_local, r << n_local)
                  for r in range(1 << g))
        assert abs(got - want) <= 1e-13 * max(1.0, float(np.sum(np.abs(op.coeffs)))), (label, got, want)
        if flag and n >= er.TABLE_TILE_BITS:
            routes, _ = er.device_routes(lay, n, 0)
            assert routes[0][0] == "V1"
            assert abs(er.emulate(lay, routes, psi, n) - want) <= 1e-13 * max(1.0, float(np.sum(np.abs(op.coeffs)))), label
