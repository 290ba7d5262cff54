"""Most probable basis states on CPU: the decision rule ``qb_top_select_pick`` through ctypes on hand-built bucket sequences, the
multi-rank logic of ``_ShardedLogic.top_states`` over gloo (world 2 and 4) with a NumPy shard backend that restates one pass of
``top_select_kernel`` and ``top_collect_kernel``, and the routing and validation of ``B200SamplerV2.top_states`` and
``measure_quasi_distributions(shots=None)`` with a fake engine."""
import math
import os

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import evqe_genome as og
from queasars_b200 import _native
from queasars_b200 import gate_list as gl
from queasars_b200 import primitives as pr
from queasars_b200.containers import QuasiDistribution
from queasars_b200.engine import check_top_limits, top_select_new, top_select_pick
from queasars_b200.evaluators import measure_quasi_distributions
from tests.fake_engine import FakeEngine, _state
from tests.test_frontend_planner import build_circuit
from tests.test_sharded_gloo import NumpyShardBackend, _free_port

ALL = ~np.uint64(0)


def oracle_top(amps, max_states, min_probability=0.0):
    """(logical indices, p) of the top states of ``amps`` in logical order: np.lexsort((k, -p)) over the eligible entries."""
    amps = np.asarray(amps, dtype=np.complex128)
    p = amps.real * amps.real + amps.imag * amps.imag
    k = np.arange(p.size, dtype=np.int64)
    ok = (p > 0) & (p >= min_probability)
    k, p = k[ok], p[ok]
    order = np.lexsort((k, -p))[:max_states]
    return k[order], p[order]


def prob_keys(p):
    return ~np.ascontiguousarray(p, dtype=np.float64).view(np.uint64)


def _logical(k, positions):
    out = np.zeros_like(k)
    for q, pos in enumerate(positions):
        out |= ((k >> np.uint64(pos)) & np.uint64(1)) << np.uint64(q)
    return out


def _shard(arr, index_offset):
    arr = np.asarray(arr, dtype=np.complex128)
    k = np.arange(arr.size, dtype=np.uint64) | np.uint64(index_offset)
    p = arr.real * arr.real + arr.imag * arr.imag
    return k, p, prob_keys(p)


def select_pass(arr, index_offset, min_probability, sel, positions):
    """One pass of top_select_kernel over one shard: bucket counts [256] of the pass ``sel`` describes."""
    k, p, key = _shard(arr, index_offset)
    ok = (p > 0) & (p >= min_probability)
    if sel.p_free > 0:
        if sel.p_free < 64:
            ok &= (key >> np.uint64(sel.p_free)) == np.uint64(sel.p_prefix)
        d = (key >> np.uint64(sel.p_free - 8)) & np.uint64(255)
    else:
        logical = _logical(k, positions)
        lo = max(0, sel.idx_hi - 8)
        ok &= (key == np.uint64(sel.p_prefix)) & ((logical >> np.uint64(sel.idx_hi)) == np.uint64(sel.idx_prefix >> sel.idx_hi))
        d = (logical >> np.uint64(lo)) & np.uint64((1 << (sel.idx_hi - lo)) - 1)
    return np.bincount(d[ok].astype(np.int64), minlength=256).astype(np.uint64)


def collect(arr, index_offset, min_probability, sel, positions, capacity):
    """top_collect_kernel over one shard: (physical indices, p) up to the stop key, in index order."""
    k, p, key = _shard(arr, index_offset)
    logical = _logical(k, positions)
    ok = (p > 0) & (p >= min_probability)
    ok &= (key < np.uint64(sel.stop_key)) | ((key == np.uint64(sel.stop_key)) & (logical <= np.uint64(sel.stop_index)))
    assert np.count_nonzero(ok) <= capacity
    return k[ok].astype(np.int64), p[ok]


class TopShardBackend(NumpyShardBackend):
    def top_select(self, state, n_local, index_offset, min_probability, sel, positions):
        return select_pass(state.numpy(), index_offset, min_probability, sel, positions)

    def top_collect(self, state, n_local, index_offset, min_probability, sel, positions, capacity):
        return collect(state.numpy(), index_offset, min_probability, sel, positions, capacity)


def run_select(arr, max_states, min_probability=0.0, positions=None):
    """The whole select + collect on one unsharded array through qb_top_select_pick -> (indices, p, passes)."""
    n = int(arr.size).bit_length() - 1
    positions = list(range(n)) if positions is None else positions
    sel = top_select_new(n, max_states)
    while not sel.done:
        top_select_pick(sel, select_pass(arr, 0, min_probability, sel, positions))
    k, p = collect(arr, 0, min_probability, sel, positions, sel.selected)
    assert k.size == sel.selected
    logical = _logical(k.astype(np.uint64), positions).astype(np.int64)
    order = np.lexsort((logical, -p))
    return logical[order], p[order], sel.passes


# ------------------------------------------------------------------ the decision rule on hand-built bucket sequences
def _counts(**buckets):
    c = np.zeros(256, dtype=np.uint64)
    for b, v in buckets.items():
        c[int(b[1:])] = v
    return c


def test_pick_takes_everything_when_fewer_entries_are_eligible():
    sel = top_select_new(10, 50)
    top_select_pick(sel, _counts(b192=30, b193=12))
    assert sel.done and sel.selected == 42 and sel.passes == 1
    assert sel.stop_key == ALL and sel.stop_index == ALL


def test_pick_every_entry_filtered_out():
    sel = top_select_new(12, 1)
    top_select_pick(sel, np.zeros(256, dtype=np.uint64))
    assert sel.done and sel.selected == 0 and sel.passes == 1
    with pytest.raises(_native.QbError):  # a finished select takes no further pass
        top_select_pick(sel, np.zeros(256, dtype=np.uint64))


def test_pick_early_exit_on_a_bucket_boundary():
    sel = top_select_new(20, 10)
    top_select_pick(sel, _counts(b192=4, b193=6, b200=1000))  # 4 + 6 == 10: bucket 193 is taken whole
    assert sel.done and sel.selected == 10 and sel.passes == 1
    assert sel.stop_key == (193 << 56) | ((1 << 56) - 1) and sel.stop_index == ALL


def test_pick_narrows_then_stops():
    sel = top_select_new(20, 10)
    top_select_pick(sel, _counts(b192=4, b193=600))
    assert not sel.done and sel.p_free == 56 and sel.p_prefix == 193 and sel.taken == 4 and sel.need == 6
    top_select_pick(sel, _counts(b7=5, b8=1, b9=594))  # 5 + 1 == 6
    assert sel.done and sel.selected == 10 and sel.stop_key == (193 << 56) | (8 << 48) | ((1 << 48) - 1)
    with pytest.raises(_native.QbError):  # a later pass whose buckets hold no more than the entries still needed is inconsistent
        bad = top_select_new(20, 10)
        top_select_pick(bad, _counts(b192=4, b193=600))
        top_select_pick(bad, _counts(b7=5))


def test_pick_cut_inside_a_run_of_ties_keeps_its_lowest_indices():
    n, key = 12, 0xC01F_0000_0000_0001
    sel = top_select_new(n, 5)
    # eight probability passes, each leaving one digit of `key` with 2 entries above and a tie run of 100 below the cut
    for j in range(8):
        digit = (key >> (56 - 8 * j)) & 255
        c = np.zeros(256, dtype=np.uint64)
        if j == 0:
            c[digit - 1], c[digit] = 2, 100
        else:
            c[digit] = 100
        top_select_pick(sel, c)
        assert not sel.done
    assert sel.p_free == 0 and sel.p_prefix == key and sel.taken == 2 and sel.need == 3 and sel.idx_hi == n
    # logical index digit of bits [4, 12): buckets 0..5 hold 1, 1, 0, 7, ... entries; the cut (3 more) falls inside bucket 3
    top_select_pick(sel, _counts(b0=1, b1=1, b3=7, b9=91))
    assert not sel.done and sel.idx_hi == 4 and sel.idx_prefix == 3 << 4 and sel.taken == 4 and sel.need == 1
    top_select_pick(sel, _counts(b2=1, b5=1, b6=5))  # the lowest index of the run, bucket 2, is the one kept
    assert sel.done and sel.selected == 5 and sel.stop_key == key and sel.stop_index == (3 << 4) | 2
    assert sel.passes == 10


def test_limits_are_validated():
    for bad in (0, -1, (1 << 20) + 1, 2.5, True):
        with pytest.raises(ValueError):
            check_top_limits(bad, 0.0)
    for bad in (-1e-300, math.nan, math.inf):
        with pytest.raises(ValueError):
            check_top_limits(4, bad)
    assert check_top_limits(np.int64(1 << 20), 0) == (1 << 20, 0.0)
    with pytest.raises(_native.QbError):
        top_select_new(10, 0)
    with pytest.raises(_native.QbError):
        top_select_new(64, 10)


# ------------------------------------------------------------------ the whole select on one array against the oracle
def _tie_state(n, seed):
    """A state with exact tie runs: a random product state whose qubits in a random half are in |+> (equal magnitudes)."""
    rng = np.random.default_rng(seed)
    amps = np.ones(1, dtype=np.complex128)
    for q in range(n):
        a = np.array([1.0, 1.0]) / np.sqrt(2.0) if rng.random() < 0.5 else np.array([np.cos(t := rng.uniform(0, np.pi)), np.sin(t) * np.exp(1j * rng.uniform(0, 6))])
        amps = np.kron(a, amps)
    return amps


@pytest.mark.parametrize("seed", range(4))
def test_select_matches_the_oracle_on_one_array(seed):
    rng = np.random.default_rng(seed)
    n = 10
    states = [_tie_state(n, seed), rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n), np.zeros(1 << n, dtype=complex)]
    states[2][[5, 17, 900]] = [0.5, 0.5, 1 / np.sqrt(2)]
    positions = list(rng.permutation(n))
    for amps in states:
        p = amps.real * amps.real + amps.imag * amps.imag
        for m in (1, 3, 7, 100, 1024, 1029):
            for min_p in (0.0, float(np.sort(p)[-min(m, p.size)]), 2.0):
                want = oracle_top(amps, m, min_p)
                got = run_select(amps, m, min_p)
                assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), (seed, m, min_p)
                # the same select with the logical bits at permuted physical positions
                phys = np.empty_like(amps)
                phys[_logical(np.arange(amps.size, dtype=np.uint64), [int(x) for x in np.argsort(positions)]).astype(np.int64)] = amps
                got = run_select(phys, m, min_p, positions=[int(x) for x in positions])
                assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), (seed, m, min_p, "permuted")


# ------------------------------------------------------------------ several ranks over gloo
CASES = ((1, 0.0), (3, 0.0), (7, 0.0), (50, 0.0), (1 << 12, 0.0), (20, 1e-3), (5, 2.0))


def _tie_circuit(n, seed):
    """|+> on a random half of the qubits and random rotations on the others (a product state with runs of exactly tied
    probabilities), applied top qubit first: the rank bits are targeted, so the state is swapped."""
    rng = np.random.default_rng(seed)
    instr = []
    for q in range(n - 1, -1, -1):
        plus = rng.random() < 0.5
        instr.append(("u", [q], [np.pi / 2, 0.0, np.pi] if plus else [float(rng.uniform(0, np.pi)), 0.0, float(rng.uniform(0, 6))]))
    return instr, []


def _worker(rank, world, port, cases, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from queasars_b200.sharded import ShardedStatevector

        results = []
        for kind, n, seed in cases:
            if kind == "evqe":
                genome, values = og.random_individual(n, 4, True, seed)
                instr = og.individual_circuit(genome, values)
            else:
                instr, values = _tie_circuit(n, seed)
            sv = ShardedStatevector(n, backend=TopShardBackend(), min_local=4)
            sv.run(gl.from_circuit(build_circuit(instr, n)), values)
            full = sv.gather_logical()
            got = [tuple(a.tolist() for a in sv.top_states(m, min_p)) for m, min_p in CASES]
            results.append((list(sv.position), full, got))
        out.put((rank, results))
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
@pytest.mark.parametrize("world", [2, 4])
def test_gloo_top_states_match_the_oracle(world):
    cases = [("evqe", 8, 11), ("evqe", 10, 12), ("ties", 9, 13), ("ties", 10, 14)]
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, cases, out)) for r in range(world)]
    [p.start() for p in procs]
    got = dict(out.get(timeout=240) for _ in range(world))
    [p.join(60) for p in procs]
    assert all(p.exitcode == 0 for p in procs)
    for r in range(1, world):  # every rank took the same decisions
        assert repr([g[2] for g in got[r]]) == repr([g[2] for g in got[0]])
    moved = cut_in_ties = 0
    for (kind, n, seed), (position, full, per_case) in zip(cases, got[0]):
        moved += position != list(range(n))
        p = full.real * full.real + full.imag * full.imag
        for (m, min_p), (idx, probs) in zip(CASES, per_case):
            want = oracle_top(full, m, min_p)
            assert idx == want[0].tolist() and probs == want[1].tolist(), (kind, n, seed, m, min_p)
            if 0 < len(probs) == m and np.count_nonzero(p == probs[-1]) > probs.count(probs[-1]):
                cut_in_ties += 1
    assert moved  # logical bits were read from permuted physical positions
    assert cut_in_ties  # at least one cut fell inside a run of ties


# ------------------------------------------------------------------ routing and validation of the primitives
class TopFakeEngine(FakeEngine):
    def __init__(self, device=0, dtype="complex128"):
        super().__init__(device, dtype)
        self.calls = []

    def top_states(self, plans, params, max_states, min_probability=0.0):
        self.calls.append(("top", len(plans), max_states, min_probability))
        return [oracle_top(_state(self._plans[pl.plan_id], np.asarray(v, dtype=np.float64).reshape(-1)), max_states, min_probability)
                for pl, v in zip(plans, params)]


class _FakeSharded:
    def __init__(self):
        self.calls = []

    def reset(self):
        pass

    def run(self, gates, values):
        self.amps = _state(gates, np.asarray(values, dtype=np.float64))

    def top_states(self, max_states, min_probability=0.0):
        self.calls.append(("top", max_states, min_probability))
        return oracle_top(self.amps, max_states, min_probability)


def _circuit(n, seed):
    genome, values = og.random_individual(n, 3, True, seed)
    return build_circuit(og.individual_circuit(genome, values), n), list(values), og.individual_circuit(genome, values)


@pytest.fixture
def fake_engines(monkeypatch):
    made = {}
    monkeypatch.setattr(pr, "get_engine", lambda device=0, dtype="complex128": made.setdefault((device, dtype), TopFakeEngine(device, dtype)))
    monkeypatch.setattr(pr._native, "device_count", lambda: 2)
    return made


@pytest.mark.parametrize("coalesce", [False, True])
def test_sampler_top_states_and_exact_quasi_distributions(fake_engines, coalesce):
    n = 5
    circ, values, _ = _circuit(n, 3)
    circ2, values2, _ = _circuit(n, 4)
    smp = pr.B200SamplerV2(devices="all", coalesce=coalesce)
    got = smp.top_states([circ, circ2, circ], [values, values2, values], 4, 0.01)
    assert len(got) == 3
    for (idx, probs), (c, v) in zip(got, [(circ, values), (circ2, values2), (circ, values)]):
        want = oracle_top(_state(gl.from_circuit(c.assign_parameters(v)), []), 4, 0.01)
        assert np.array_equal(idx, want[0]) and np.allclose(probs, want[1], rtol=1e-12, atol=0)
    assert {c[2:] for e in fake_engines.values() for c in e.calls} == {(4, 0.01)}
    dists = measure_quasi_distributions([circ, circ2], [values, values2], smp, None, max_states=3)
    assert all(isinstance(d, QuasiDistribution) and d.shots is None and len(d) == 3 for d in dists)
    idx, probs = got[1]
    assert list(dists[1].keys()) == list(idx[:3]) and list(dists[1].values()) == list(probs[:3])
    assert len(measure_quasi_distributions([circ], [values], smp, None)[0]) == 1 << n  # max_states=1024 holds all 32 entries
    with pytest.raises(ValueError):
        smp.top_states([circ], [values], 0)
    with pytest.raises(ValueError):
        smp.top_states([circ], [values], 1 << 21)
    with pytest.raises(ValueError):
        smp.top_states([circ], [values], 4, -0.5)
    with pytest.raises(ValueError):
        smp.top_states([circ], [values], 4, math.nan)
    with pytest.raises(ValueError):
        smp.top_states([circ], [values, values], 4)
    with pytest.raises(ValueError):
        smp.top_states([circ, _circuit(n + 1, 5)[0]], [values, _circuit(n + 1, 5)[1]], 4)
    with pytest.raises(ValueError):
        measure_quasi_distributions([circ], [values], smp, None, max_states=0)
    assert smp.top_states([], [], 4) == []


def test_sampler_top_states_route_sharded_widths_on_one_device(fake_engines, monkeypatch):
    n = 5
    circ, values, _ = _circuit(n, 6)
    fake = _FakeSharded()
    smp = pr.B200SamplerV2(shard_min_qubits=n, coalesce=False)  # one device: the sharded route still runs
    monkeypatch.setattr(smp, "_sharded_state", lambda width: fake)
    got = smp.top_states([circ, circ], [values, values], 6, 0.0)
    assert fake.calls == [("top", 6, 0.0), ("top", 6, 0.0)]
    assert not any(e.calls for e in fake_engines.values())  # nothing went to the single-device engines
    want = oracle_top(_state(gl.from_circuit(circ.assign_parameters(values)), []), 6)
    assert np.array_equal(got[0][0], want[0])
    dist_ = measure_quasi_distributions([circ], [values], smp, None, max_states=2)[0]
    assert dist_.shots is None and list(dist_) == list(want[0][:2])


def test_shots_none_with_a_foreign_sampler_keeps_the_generic_path():
    class Foreign:
        def __init__(self):
            self.shots = "unset"

        def run(self, pubs, shots=None):
            self.shots = shots
            raise RuntimeError("generic path")

    class Circ:
        def measure_all(self, inplace=False):
            return self

    s = Foreign()
    with pytest.raises(RuntimeError, match="generic path"):
        measure_quasi_distributions([Circ()], [[0.0]], s, None)
    assert s.shots is None
