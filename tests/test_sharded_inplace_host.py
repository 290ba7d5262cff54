"""Sharded statevectors with ONE buffer per shard (the in-place global <-> local exchange, ``swap_inplace_p2p_kernel``) on CPU:
a NumPy mirror of the kernel's index arithmetic, the buffer-count choice of both drivers with injected allocation outcomes, the
one-buffer routes of ``LocalShardedStatevector`` against its two-buffer routes with NumPy stand-ins for the device, and the
multi-process driver over gloo."""
import itertools
import os

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import evqe_genome as og
from oracle import qiskit_semantics as oq
from queasars_b200 import _native
from queasars_b200 import gate_list as gl
from tests.test_frontend_planner import build_circuit
from tests.test_sharded_cvar_host import ALPHAS, random_ising_masks, select_pass
from tests.test_sharded_gloo import NumpyShardBackend, _free_port

RUN_BITS = 10  # kSwapRunBits


def inplace_work(n_local, lp, rank):
    """NumPy mirror of swap_inplace_p2p_kernel (queasars_b200/csrc/qb_kernels.cuh) for one rank: item number t -> peer d and the
    pair (own index i, peer index i').  Run u = t >> run_bits goes to d = rank ^ (1 + u % (W-1)); the pair number within that peer,
    ((u // (W-1)) << run_bits) | (t & run_mask), is expanded to i by dropping in d's bits at lp and the owner bit (rank > d) at p0,
    the highest local position not in lp."""
    g = len(lp)
    world = 1 << g
    rb = min(RUN_BITS, n_local - g - 1)
    p0 = max(set(range(n_local)) - set(lp))
    ins = sorted([(p, j) for j, p in enumerate(lp)] + [(p0, g)])
    items = (world - 1) << (n_local - g - 1)
    t = np.arange(items, dtype=np.int64)
    u = t >> rb
    d = rank ^ (1 + u % (world - 1))
    bits = d | ((rank > d).astype(np.int64) << g)
    i = ((u // (world - 1)) << rb) | (t & ((1 << rb) - 1))
    for p, src in ins:
        i = ((i >> p) << (p + 1)) | (i & ((1 << p) - 1)) | (((bits >> src) & 1) << p)
    lpmask = sum(1 << p for p in lp)
    rbits = sum(((rank >> j) & 1) << p for j, p in enumerate(lp))
    return d, i, (i & ~lpmask) | rbits


def swapped_permutation(full, n_local, lp):
    """The exchange on the full vector: rank bit j <-> local bit lp[j]."""
    idx = np.arange(full.size, dtype=np.int64)
    swapped = idx.copy()
    for j, p in enumerate(lp):
        a, b = (idx >> (n_local + j)) & 1, (idx >> p) & 1
        swapped &= ~((1 << (n_local + j)) | (1 << p))
        swapped |= (b << (n_local + j)) | (a << p)
    want = np.empty_like(full)
    want[swapped] = full
    return want


LAYOUTS = [(2, [0]), (2, [1]), (10, [9]), (12, [0]), (3, [0, 2]), (11, [2, 10]), (4, [0, 1, 3]), (12, [0, 5, 11]), (12, [3, 4, 5]),
           (5, [0, 1, 2, 4]), (5, [1, 2, 3, 4]), (13, [0, 6, 7, 12]), (14, [1, 2, 3, 13])]


@pytest.mark.parametrize("n_local,lp", LAYOUTS)
def test_inplace_work_order_is_the_bit_permutation(n_local, lp):
    """Over all ranks every cross pair is handled exactly once, no fixed element is touched, the swaps give the permutation rank
    bit j <-> local bit lp[j], and at every item number the ranks target pairwise different peers.  The layouts cover g = 1..4,
    lp sets with bit 0 and bit n_local - 1, and the smallest n_local the kernel takes (g + 1)."""
    g, world, size = len(lp), 1 << len(lp), 1 << n_local
    full = np.arange(world * size, dtype=np.int64) * 7 + 3
    touched = np.zeros(world * size, dtype=np.int64)
    out = full.copy()
    peers = []
    for r in range(world):
        d, i, i2 = inplace_work(n_local, lp, r)
        assert np.all(d != r) and np.all((d >= 0) & (d < world))
        own, there = (r << n_local) | i, (d << n_local) | i2
        lp_bits = sum(((i >> p) & 1) << j for j, p in enumerate(lp))
        assert np.array_equal(lp_bits, d)  # i is a cross element bound for d
        np.add.at(touched, own, 1)
        np.add.at(touched, there, 1)
        out[own], out[there] = full[there], full[own]
        peers.append(d)
    idx = np.arange(world * size, dtype=np.int64)
    home = sum(((idx >> p) & 1) << j for j, p in enumerate(lp))
    cross = home != (idx >> n_local)
    assert np.all(touched[cross] == 1) and np.all(touched[~cross] == 0)
    assert np.array_equal(out, swapped_permutation(full, n_local, lp))
    stacked = np.stack(peers)  # ranks x item numbers
    for k in range(stacked.shape[1]):
        assert len(set(stacked[:, k].tolist())) == world


def test_every_rank_moves_half_of_its_cross_elements_to_every_peer():
    n_local, lp = 12, [0, 5, 11]
    for r in range(8):
        d, _, _ = inplace_work(n_local, lp, r)
        counts = np.bincount(d, minlength=8)
        assert counts[r] == 0 and np.all(np.delete(counts, r) == (1 << (n_local - 3)) // 2)


# ---------------------------------------------------------------------------------------------------- NumPy stand-ins for the device
MEMORY: dict = {}
_ADDRESSES = itertools.count(1 << 20, 1 << 20)


class FakeEngine:
    """Device memory = NumPy arrays in MEMORY; ``fail_at`` = the allocation number (1-based) from which device_alloc fails with
    ``code``."""

    def __init__(self, device=0, fail_at=None, code=_native.QB_ERR_MEMORY):
        self.device, self.fail_at, self.code = device, fail_at, code
        self.allocs, self.freed = 0, []

    def enable_peer_access(self, peer):
        pass

    def synchronize(self):
        pass

    def device_alloc(self, nbytes):
        self.allocs += 1
        if self.fail_at is not None and self.allocs >= self.fail_at:
            raise _native.QbError(self.code, "injected")
        ptr = next(_ADDRESSES)
        MEMORY[ptr] = np.zeros(nbytes // 16, dtype=np.complex128)
        return ptr

    def device_free(self, ptr):
        self.freed.append(ptr)
        MEMORY.pop(ptr, None)

    def device_read(self, ptr, offset, out):
        out[:] = MEMORY[ptr][offset // 16 : offset // 16 + out.size]
        return out

    def ipc_export(self, ptr):
        return int(ptr).to_bytes(64, "little")

    def ipc_open(self, handle):
        return int.from_bytes(handle, "little") + (1 << 50)  # a different address for the same buffer

    def ipc_close(self, ptr):
        pass


class _View:
    def __init__(self, arr):
        self.arr = arr

    def numpy(self):
        return self.arr


class PointerBackend(NumpyShardBackend):
    """The shard backend on device addresses (MEMORY), with both exchange kernels restated in NumPy."""

    def __init__(self):
        self.select_calls = []
        self.inplace_calls = 0

    def apply(self, state, *args):
        super().apply(_View(MEMORY[state]), *args)

    def diagonal_expectation(self, state, *args):
        return super().diagonal_expectation(_View(MEMORY[state]), *args)

    def pauli_expectation(self, state, *args):
        return super().pauli_expectation(_View(MEMORY[state]), *args)

    def sample(self, state, *args):
        return super().sample(_View(MEMORY[state]), *args)

    def cvar_select(self, state, cache, cache_mode, z_masks, coeffs, n_total, n_local, index_offset, spec):
        self.select_calls.append((cache, cache_mode))
        return select_pass(MEMORY[state], z_masks, coeffs, index_offset, spec)

    def swap_p2p(self, state, dst, n_local, rank, lp):
        src = MEMORY[state]
        i = np.arange(src.size, dtype=np.int64)
        d = sum(((i >> p) & 1) << j for j, p in enumerate(lp))
        rbits = sum(((rank >> j) & 1) << p for j, p in enumerate(lp))
        to = (i & ~sum(1 << p for p in lp)) | rbits
        for peer in range(len(dst)):
            MEMORY[dst[peer]][to[d == peer]] = src[d == peer]

    def swap_inplace_p2p(self, state, states, n_local, rank, lp):
        self.inplace_calls += 1
        d, i, i2 = inplace_work(n_local, lp, rank)
        own = MEMORY[states[rank]]
        for peer in set(d.tolist()):
            sel = d == peer
            there = MEMORY[states[peer]]
            a, b = own[i[sel]].copy(), there[i2[sel]].copy()
            own[i[sel]], there[i2[sel]] = b, a


def local_state(n, world, buffers, engines=None):
    from queasars_b200.sharded import LocalShardedStatevector

    sv = LocalShardedStatevector(n, engines or [FakeEngine() for _ in range(world)], min_local=3, buffers=buffers)
    sv.backends = [PointerBackend() for _ in range(world)]
    return sv


def test_buffers_none_takes_two_and_falls_back_to_one_on_out_of_memory():
    sv = local_state(8, 2, None)
    assert sv.buffers == 2 and sv.describe()["buffers"] == 2 and sv.swap_path.startswith("swap_p2p_kernel")
    sv.close()
    engines = [FakeEngine(), FakeEngine(fail_at=2)]  # the second shard's second buffer does not fit
    sv = local_state(8, 2, None, engines)
    assert sv.buffers == 1 and len(sv._bufs) == 1 and sv.swap_path.startswith("swap_inplace_p2p_kernel")
    assert len(engines[0].freed) == 1  # the first shard's second buffer was freed again
    live = [b.ptr for b in sv._bufs[0]]
    assert all(p in MEMORY for p in live)
    sv.close()


@pytest.mark.parametrize("buffers,code", [(None, _native.QB_ERR_CUDA), (2, _native.QB_ERR_MEMORY)])
def test_other_errors_and_forced_two_buffers_are_raised(buffers, code):
    engines = [FakeEngine(), FakeEngine(fail_at=2, code=code)]
    with pytest.raises(_native.QbError) as info:
        local_state(8, 2, buffers, engines)
    assert info.value.code == code
    assert len(engines[0].freed) == 2 and len(engines[1].freed) == 1  # nothing stays allocated


def test_buffers_one_allocates_one_set_and_bad_values_are_refused():
    engines = [FakeEngine(fail_at=2) for _ in range(4)]
    sv = local_state(9, 4, 1, engines)
    assert sv.buffers == 1 and all(e.allocs == 1 for e in engines)
    sv.close()
    with pytest.raises(ValueError):
        local_state(9, 4, 3)


@pytest.mark.parametrize("n,world,layers,seed", [(8, 2, 4, 0), (9, 4, 5, 1), (10, 8, 3, 2)])
def test_one_buffer_routes_equal_the_two_buffer_routes(n, world, layers, seed):
    """The whole host logic with the kernels restated in NumPy: states, placements, swaps, <H>, Pauli sums, samples and CVaR of
    the one-buffer driver are bit-identical to the two-buffer driver's, and the one-buffer CVaR never passes a cache."""
    from queasars_b200.operators import SparsePauliOp

    genome, values = og.random_individual(n, layers, True, seed)
    instr = og.individual_circuit(genome, values)
    gates = gl.from_circuit(build_circuit(instr, n))
    z, c = random_ising_masks(n, 70 + seed)
    labels = [("X" + "I" * (n - 2) + "Z", 0.7), ("Z" * n, 0.25), ("I" * (n - 1) + "Y", -0.4)]  # X on the top qubit flips a rank bit
    uniforms = np.random.default_rng(seed).random(500)
    results = {}
    for buffers in (2, 1):
        sv = local_state(n, world, buffers)
        sv.run(gates, values)
        assert sv.swaps_done >= 1
        out = [sv.gather_physical().tobytes(), list(sv.position), sv.swaps_done, sv.bytes_sent]
        out.append(sv.diagonal_expectation(z, c))
        out.append(sv.expectation(SparsePauliOp.from_list(labels)))
        out += [list(sv.position), sv.swaps_done, sv.sample(500, uniforms=uniforms).tolist()]
        out.append([sv.cvar(z, c, a) for a in ALPHAS])
        out.append([sv.cvar(z, c, a, cache=False) for a in ALPHAS])
        calls = [call for b in sv.backends for call in b.select_calls]
        if buffers == 1:
            assert calls and all(cache is None and mode == 0 for cache, mode in calls)
            assert sum(b.inplace_calls for b in sv.backends) == world * sv.swaps_done
        else:
            assert any(mode == 1 for _, mode in calls) and any(mode == 2 for _, mode in calls)
        results[buffers] = out
        want = oq.statevector(instr, n, values)
        sv2 = local_state(n, world, buffers)
        sv2.run(gates, values)
        assert np.max(np.abs(sv2.gather_logical() - want)) < 1e-12
        sv.close(), sv2.close()
    assert repr(results[1]) == repr(results[2])


# ---------------------------------------------------------------------------------------------------- multi-process driver over gloo
def _worker(rank, world, port, mode, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from queasars_b200.sharded import ShardedStatevector

        if mode == "one buffer without peer mapping":
            try:
                ShardedStatevector(8, backend=NumpyShardBackend(), min_local=4, buffers=1)
                out.put((rank, None))
            except ValueError as exc:
                out.put((rank, str(exc)))
        elif mode == "none keeps the staged route":
            n = 8
            genome, values = og.random_individual(n, 4, True, 5)
            instr = og.individual_circuit(genome, values)
            sv = ShardedStatevector(n, backend=NumpyShardBackend(), min_local=4)
            sv.run(gl.from_circuit(build_circuit(instr, n)), values)
            err = float(np.max(np.abs(sv.gather_logical() - oq.statevector(instr, n, values))))
            out.put((rank, (sv.buffers, sv.spare is not None, sv.swaps_done >= 1, err, sv.describe()["swap_path"])))
        else:  # collective buffer count with injected allocation outcomes
            sv = ShardedStatevector(8, backend=NumpyShardBackend(), min_local=4)
            fail_second = rank == world - 1
            rows = []
            for buffers in (None, 2, 1):
                engine = FakeEngine(fail_at=2 if fail_second else None)
                sv.backend = type("B", (), {"engine": engine})()
                sv.swap_fallback_reason = None
                got = sv._map_ipc_buffers(1 << sv.n_local, buffers)
                if got is None:
                    rows.append((buffers, None, len(engine.freed), engine.allocs, sv.swap_fallback_reason is not None))
                else:
                    bufs, peer = got
                    rows.append((buffers, len(bufs), len(engine.freed), engine.allocs, [p[rank] == bufs[i].ptr for i, p in enumerate(peer)]))
                    for b in bufs:
                        b.free()
                    sv._mapped = []
            out.put((rank, rows))
    finally:
        dist.destroy_process_group()


def _run(world, mode):
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, mode, out)) for r in range(world)]
    [p.start() for p in procs]
    got = dict(out.get(timeout=120) for _ in range(world))
    [p.join(60) for p in procs]
    assert all(p.exitcode == 0 for p in procs)
    return got


def test_gloo_one_buffer_without_peer_mapping_raises_on_every_rank():
    got = _run(2, "one buffer without peer mapping")
    assert all(msg is not None and "peer-mapped memory" in msg for msg in got.values())
    assert got[0] == got[1]


def test_gloo_buffers_none_runs_the_two_buffer_staged_route():
    got = _run(2, "none keeps the staged route")
    for buffers, has_spare, swapped, err, path in got.values():
        assert buffers == 2 and has_spare and swapped and err < 1e-12 and path == "pack + all_to_all_single + unpack"


def test_gloo_buffer_count_is_collective():
    """Only the last rank's second allocation fails: with None every rank takes one buffer (the others free their second); with
    buffers=2 every rank gives up the peer mapping; with 1 nobody tries a second allocation."""
    world = 2
    got = _run(world, "collective")
    for rank, rows in got.items():
        last = rank == world - 1
        (b0, n0, freed0, allocs0, own0), (b1, n1, freed1, _, reason1), (b2, n2, freed2, allocs2, own2) = rows
        assert b0 is None and n0 == 1 and own0 == [True]
        assert freed0 == (0 if last else 1) and allocs0 == 2
        assert b1 == 2 and n1 is None and reason1 and freed1 == (1 if last else 2)  # every rank released what it had allocated
        assert b2 == 1 and n2 == 1 and allocs2 == 1 and freed2 == 0
