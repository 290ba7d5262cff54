"""Exact (shot-free) CVaR of a sharded statevector on CPU: the multi-rank select logic of ``_ShardedLogic.cvar`` over gloo (world
2 and 4) with a NumPy shard backend that restates one select pass of ``cvar_select_kernel``, the energy key transform, and the
routing of ``B200SamplerV2`` at sharded widths."""
import os

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import evqe_genome as og
from oracle import qiskit_semantics as oq
from queasars_b200 import expectation as ex
from queasars_b200 import gate_list as gl
from queasars_b200 import primitives as pr
from queasars_b200.operators import SparsePauliOp
from queasars_b200.sharded import energy_from_key, energy_keys
from tests.test_frontend_planner import build_circuit
from tests.test_sharded_gloo import NumpyShardBackend, _free_port

ALPHAS = (0.05, 0.25, 0.5, 0.9, 1.0)


def select_pass(arr, z_masks, coeffs, index_offset, spec):
    """One select pass over one shard, as cvar_select_kernel computes it (sums in index order instead of the kernel's order)."""
    e_prefix, e_free, digit_kind, positions, idx_mask, idx_value = spec
    k = np.arange(arr.size, dtype=np.uint64) | np.uint64(index_offset)
    p = arr.real**2 + arr.imag**2
    e = np.zeros(arr.size)
    for z, c in zip(z_masks, coeffs):  # diag_table_kernel's loop: start at 0.0, add +-c in term order
        e = e + np.where(np.bitwise_count(k & np.uint64(z)) & 1, -c, c)
    key = energy_keys(e)
    ok = (k & np.uint64(idx_mask)) == np.uint64(idx_value)
    if e_free < 64:
        ok &= (key >> np.uint64(e_free)) == np.uint64(e_prefix)
    if digit_kind == 0:
        d = (key >> np.uint64(e_free - 8)) & np.uint64(255)
    else:
        d = np.zeros(arr.size, dtype=np.uint64)
        for j, pos in enumerate(positions):
            d |= ((k >> np.uint64(pos)) & np.uint64(1)) << np.uint64(j)
    d = d[ok].astype(np.int64)
    sums = np.stack([np.bincount(d, weights=p[ok], minlength=256), np.bincount(d, weights=(p * e)[ok], minlength=256)])
    ints = np.zeros((4, 256), dtype=np.uint64)
    ints[0] = np.bincount(d, minlength=256)
    ints[1] = ~np.uint64(0)
    ints[3] = ~np.uint64(0)
    np.minimum.at(ints[1], d, key[ok])
    np.maximum.at(ints[2], d, key[ok])
    np.minimum.at(ints[3], d, k[ok])
    return sums, ints


class SelectShardBackend(NumpyShardBackend):
    def cvar_select(self, state, cache, cache_mode, z_masks, coeffs, n_total, n_local, index_offset, spec):
        return select_pass(state.numpy(), z_masks, coeffs, index_offset, spec)


def random_ising_masks(n, seed):
    rng = np.random.default_rng(seed)
    z = [1 << q for q in range(n)] + [(1 << q) | (1 << ((q + 1) % n)) for q in range(n)]
    return z, [float(c) for c in rng.normal(size=len(z))]


def jssp_masks(entry):
    z, c = ex.merge_diagonal_terms(np.asarray(entry["z_masks"], dtype=np.uint64), np.asarray(entry["coeffs"], dtype=np.float64))
    return [int(v) for v in z], [float(v) for v in c]


def oracle_stop(probs, energies, alpha):
    """(value, basis index of the stop entry, size of the stop entry's run of tied energies, knife edge?)"""
    value = ex.lower_tail_expectation_arrays(probs, energies, alpha)
    order = np.arange(probs.size) if ex._close(alpha, 1) else np.argsort(energies, kind="stable")
    cum = np.cumsum(probs[order])
    bound = alpha - (1e-8 + 1e-5 * alpha)
    stop = int(np.nonzero(cum >= bound)[0][0])
    before = np.concatenate(([0.0], cum[:-1]))
    edge = int(np.count_nonzero((before < bound + 1e-12) & (cum >= bound - 1e-12))) > 1
    ties = int(np.count_nonzero(energies == energies[order[stop]]))
    return value, int(order[stop]), ties, edge


def _worker(rank, world, port, cases, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from queasars_b200.sharded import ShardedStatevector

        results = []
        for n, layers, seed, z, c in cases:
            genome, values = og.random_individual(n, layers, True, seed)
            instr = og.individual_circuit(genome, values)
            sv = ShardedStatevector(n, backend=SelectShardBackend(), min_local=4)
            sv.run(gl.from_circuit(build_circuit(instr, n)), values)
            results.append((list(sv.position), [sv.cvar(z, c, alpha) for alpha in ALPHAS]))
        out.put((rank, results))
    finally:
        dist.destroy_process_group()


def _cases(jssp_golden):
    cases = []
    for n, seed in ((8, 0), (9, 1), (10, 2)):
        z, c = random_ising_masks(n, 50 + seed)
        cases.append((n, 4, 300 + seed, z, c))
    for name, seed in (("jssp_8q", 7), ("jssp_unit_test", 8)):
        z, c = jssp_masks(jssp_golden[name])
        cases.append((int(jssp_golden[name]["n_qubits"]), 4, 400 + seed, z, c))
    return cases


@pytest.mark.timeout(300)
@pytest.mark.parametrize("world", [2, 4])
def test_gloo_select_matches_the_oracle(world, jssp_golden):
    cases = _cases(jssp_golden)
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, cases, out)) for r in range(world)]
    [p.start() for p in procs]
    got = dict(out.get(timeout=240) for _ in range(world))
    [p.join(60) for p in procs]
    assert all(p.exitcode == 0 for p in procs)
    for r in range(1, world):  # every rank took the same decisions: bit-identical values and stop indices
        assert repr(got[r]) == repr(got[0])
    inside_ties = 0
    moved = 0
    for (n, layers, seed, z, c), (position, per_alpha) in zip(cases, got[0]):
        moved += position != list(range(n))
        genome, values = og.random_individual(n, layers, True, seed)
        probs = np.abs(oq.statevector(og.individual_circuit(genome, values), n, values)) ** 2
        energies = oq.diagonal_table(n, list(zip(z, c)))
        for alpha, (value, stop) in zip(ALPHAS, per_alpha):
            want, want_stop, ties, edge = oracle_stop(probs, energies, alpha)
            if edge:
                continue
            assert abs(value - want) <= 1e-12 * max(1.0, abs(want)), (n, seed, alpha)
            assert stop == want_stop, (n, seed, alpha)
            inside_ties += ties > 1 and not ex._close(alpha, 1)
    assert moved  # the circuits leave a non-identity qubit placement: logical bits are read from permuted positions
    assert inside_ties  # at least one stop inside a run of tied energies: the order within the tie is checked


def test_single_rank_select_and_lower_tail_without_mass():
    from queasars_b200.sharded import ShardedStatevector

    n = 6
    genome, values = og.random_individual(n, 3, True, 9)
    instr = og.individual_circuit(genome, values)
    sv = ShardedStatevector(n, backend=SelectShardBackend(), min_local=4)
    sv.run(gl.from_circuit(build_circuit(instr, n)), values)
    z, c = random_ising_masks(n, 4)
    probs = np.abs(oq.statevector(instr, n, values)) ** 2
    energies = oq.diagonal_table(n, list(zip(z, c)))
    for alpha in ALPHAS:
        value, stop = sv.cvar(z, c, alpha)
        want, want_stop, _, _ = oracle_stop(probs, energies, alpha)
        assert value == pytest.approx(want, rel=1e-12, abs=1e-12) and stop == want_stop
    # duplicate terms are merged like the device Hamiltonian's
    assert sv.cvar(z + z[:3], c + c[:3], 0.3)[0] == pytest.approx(
        ex.lower_tail_expectation_arrays(probs, oq.diagonal_table(n, list(zip(z, [ci * (2 if i < 3 else 1) for i, ci in enumerate(c)]))), 0.3), rel=1e-12)
    with pytest.raises(ValueError):
        sv.cvar(z, c, 0.0)


def test_energy_key_is_monotone_with_signed_zeros_tied():
    rng = np.random.default_rng(1)
    vals = np.concatenate([rng.normal(size=2000) * 10.0 ** rng.integers(-300, 300, 2000), [0.0, -0.0, np.inf, -np.inf, 5e-324, -5e-324,
                                                                                        np.finfo(float).max, -np.finfo(float).max]])
    keys = energy_keys(vals)
    order = np.argsort(vals, kind="stable")
    assert np.all(np.diff(keys[order].astype(object)) >= 0)  # ascending energies -> non-decreasing keys
    for a, b in zip(vals[order][:-1], vals[order][1:]):
        ka, kb = energy_keys([a])[0], energy_keys([b])[0]
        assert (ka == kb) == (a == b) and (ka < kb) == (a < b)
    assert energy_keys([-0.0])[0] == energy_keys([0.0])[0]
    assert np.array_equal(np.argsort(keys, kind="stable"), order)
    for v in vals[np.isfinite(vals)][:50]:
        back = energy_from_key(energy_keys([v])[0])
        assert back == v and (v != 0 or np.signbit(back) is np.False_)


class _FakeSharded:
    def __init__(self, n):
        self.n, self.calls = n, []

    def reset(self):
        pass

    def run(self, gates, values):
        self.state = (gates, np.asarray(values))

    def cvar(self, z, c, alpha):
        self.calls.append(("cvar", alpha))
        return 1.5, 0

    def diagonal_expectation(self, z, c):
        self.calls.append(("exp",))
        return 2.5


def test_sampler_routes_sharded_widths(monkeypatch):
    from tests.test_cvar_exact_host import CvarFakeEngine, case, ising

    made = {}
    monkeypatch.setattr(pr, "get_engine", lambda device=0, dtype="complex128": made.setdefault((device, dtype), CvarFakeEngine(device, dtype)))
    monkeypatch.setattr(pr._native, "device_count", lambda: 2)
    n = 4
    op = SparsePauliOp.from_list(ising(n))
    _, values, circ = case(n, 2, 1)
    fake = _FakeSharded(n)
    smp = pr.B200SamplerV2(devices="all", shard_min_qubits=n, coalesce=False)
    monkeypatch.setattr(smp, "_sharded_state", lambda width: fake)
    assert list(smp.cvar_values([circ, circ], [values, values], op, 0.4)) == [1.5, 1.5]
    assert list(smp._exact("exp", [circ], [values], op, 1.0)) == [2.5]
    assert fake.calls == [("cvar", 0.4), ("cvar", 0.4), ("exp",)]
    assert not any(c for e in made.values() for c in e.calls)  # nothing went to the single-device engines
    with pytest.raises(ValueError):
        smp.cvar_values([circ], [values], SparsePauliOp.from_list([("XIIZ", 1.0)]), 0.5)
    one = pr.B200SamplerV2(shard_min_qubits=n)
    with pytest.raises(NotImplementedError):
        one.cvar_values([circ], [values], op, 0.5)
