"""Which kernels reduce a state to <H> for one operator, a NumPy emulator of those kernels, and operators that reach all of
them.  Test infrastructure.

``hamiltonian_layout`` restates what ``Engine.hamiltonian`` and ``qb_hamiltonian_create`` (csrc/qb_api.cu) build for an
operator: duplicate strings merged (``engine.merge_duplicate_terms``), x-mask groups in first-appearance order with the diagonal
group first, weights ``w = c * i^{#Y}``, the diagonal table (for the table width ``max(n, QB_TILE_BITS)``) and the tile-sweep
plan of the non-diagonal groups (``plan_tile_sweeps``: tile qubits, ``xloc``, ``trivial``, generic groups).

``batch_routes`` restates the selection of ``launch_expectation_t`` (every batched entry point: one-shot calls, CUDA graphs of
one circuit, pipelined submissions, resident batches) and ``device_routes`` that of ``expectation_state_t``
(``qb_expectation_device``, the sharded route).  Both return the (route class, group) pairs in launch order and the number of
expectation kernels plus reductions they launch.  The element dtype selects no route.  The route classes are

  D1  diagonal part in the fused epilogue of the last sweep, state not stored (diagonal operator with a table)
  D2  the same with the state stored (other groups read it)
  D3  diagonal group on the fly, terms staged in shared memory (<= 2000)      D4  the same, terms unstaged (> 2000)
  D5  a table exists, but not for the plan's width: the diagonal group on the fly
  T1  trivial pure-X group, partner in the thread's registers (S = 1, 2, 4: flipped tile-local bit 8, 9, 10)
  T2  trivial group, partner in shared memory                                  T3  general group in a tile sweep
  G1  generic group kernel, terms staged                                       G2  the same, terms unstaged
  E0  no terms at all
  V1  table kernel on the device route            V2  diagonal group on the fly on the device route, z on rank bits
  V3  general tile group on the device route with z on rank bits
  V5  generic group of the device route with z on rank bits

and ``features`` adds what the kernels branch on beyond the class: S of T1, even / odd #Y and complex weights of T3 groups,
several tile sweeps (T4) and several groups per sweep, an unusable tile plan (T5), no tile kernel on a device route below one
tile (V4), and the number of table-builder launches.

``emulate`` evaluates a route list on a NumPy state exactly as the kernels are encoded: a tile is gathered through
``tile_qubits``, pairs are formed through ``xloc``, ``W(k)`` from the z masks and the global index (with the rank offset), and
the table is built chunk by chunk as ``fill_diag_table`` does.  ``reference`` is the plain per-term reduction the GPU tests
compare with."""
from __future__ import annotations

import dataclasses
import math

import numpy as np

from queasars_b200 import engine as qe

EXP_TILE_BITS = 11  # qb::kExpTileBits
LOW_BITS = 4  # QB_LOW_BITS
TABLE_TILE_BITS = 11  # QB_TILE_BITS: the table is built for max(n, QB_TILE_BITS) qubits
MAX_STAGED_TERMS = 2000  # kMaxStagedTerms
TABLE_TERM_CHUNK = 3000  # kTableTermChunk


class RouteError(ValueError):
    """The host refuses the operator on this route (QB_ERR_INVALID)."""


@dataclasses.dataclass
class Group:
    xmask: int
    z: np.ndarray  # uint64
    w: np.ndarray  # complex: c * i^{#Y}
    xloc: int = 0  # x mask in the tile-local bit positions of its sweep
    trivial: bool = False


@dataclasses.dataclass
class Sweep:
    tile_qubits: list
    groups: list  # group indices


@dataclasses.dataclass
class Layout:
    n: int
    groups: list
    diag_z: np.ndarray
    diag_c: np.ndarray
    table: bool
    sweeps: list
    generic: list

    @property
    def n_diag(self) -> int:
        return len(self.diag_z)

    @property
    def diagonal(self) -> bool:
        return all(g.xmask == 0 for g in self.groups)

    @property
    def table_n_eff(self) -> int:
        return max(self.n, TABLE_TILE_BITS)

    @property
    def tile_n_eff(self) -> int:
        return max(self.n, EXP_TILE_BITS)

    @property
    def table_chunks(self) -> int:
        return -(-self.n_diag // TABLE_TERM_CHUNK) if self.table else 0


def default_build_table(n_diag: int, n: int, tile_bits: int, workspace_bytes: int) -> bool:
    """``Engine.hamiltonian(build_table=None)``."""
    return n_diag > 8 and (8 << max(n, tile_bits)) <= workspace_bytes // 16


def _popcount(a):
    return np.bitwise_count(np.asarray(a, dtype=np.uint64))


def plan_tile_sweeps(n_eff: int, xmask: list, pending: list):
    """-> (sweeps, xloc per group, generic groups) of ``plan_tile_sweeps``."""
    tp_sweeps, xloc, generic = [], [0] * len(xmask), []
    pending = list(pending)
    while pending:
        tile = (1 << LOW_BITS) - 1
        chosen, rest = [], []
        for g in pending:
            want = tile | xmask[g]
            if bin(want).count("1") <= EXP_TILE_BITS:
                tile = want
                chosen.append(g)
            else:
                rest.append(g)
        if not chosen:
            generic.append(pending.pop(0))
            continue
        q = 0
        while bin(tile).count("1") < EXP_TILE_BITS:
            tile |= 1 << q
            q += 1
        qubits = [q for q in range(n_eff) if (tile >> q) & 1]
        pos = {q: i for i, q in enumerate(qubits)}
        for g in chosen:
            xloc[g] = sum(1 << pos[q] for q in range(n_eff) if (xmask[g] >> q) & 1)
        tp_sweeps.append(Sweep(qubits, chosen))
        pending = rest
    return tp_sweeps, xloc, generic


def hamiltonian_layout(n: int, x, z, c, build_table: bool) -> Layout:
    """What ``Engine.hamiltonian(op, build_table)`` uploads for the operator's (x, z, c) terms."""
    x, z, c = qe.merge_duplicate_terms(x, z, c)
    x = [int(v) for v in x]
    z = [int(v) for v in z]
    c = np.asarray(c, dtype=complex)
    xs, members = [], {}
    for t, xm in enumerate(x):
        if xm not in members:
            xs.append(xm)
            members[xm] = []
        members[xm].append(t)
    groups = []
    for xm in xs:
        ts = members[xm]
        ny = [bin(x[t] & z[t]).count("1") & 3 for t in ts]
        grp = Group(xm, np.array([z[t] for t in ts], dtype=np.uint64), np.array([c[t] * 1j ** k for t, k in zip(ts, ny)], dtype=complex))
        if xm == 0:
            groups.insert(0, grp)
        else:
            groups.append(grp)
    dts = members.get(0, [])
    diag_z = np.array([z[t] for t in dts], dtype=np.uint64)
    diag_c = np.array([c[t].real for t in dts], dtype=np.float64)
    tile_n_eff = max(n, EXP_TILE_BITS)
    sweeps, xloc, generic = plan_tile_sweeps(tile_n_eff, [g.xmask for g in groups], [i for i, g in enumerate(groups) if g.xmask])
    for i, g in enumerate(groups):
        g.xloc = xloc[i]
        g.trivial = len(g.z) == 1 and int(g.z[0]) == 0
    return Layout(n, groups, diag_z, diag_c, bool(build_table) and len(dts) > 0, sweeps, generic)


def layout_of(op, build_table: bool) -> Layout:
    n, x, z, c = qe.operator_terms(op)
    return hamiltonian_layout(n, x, z, c, build_table)


# ----------------------------------------------------------------------------------------------- routes
def _tile_class(g: Group) -> str:
    if not g.trivial:
        return "T3"
    hi = g.xloc >> 8
    return "T1" if (g.xloc & 255) == 0 and hi in (1, 2, 4) else "T2"


def _staged(g: Group) -> bool:
    return len(g.z) <= MAX_STAGED_TERMS


def batch_routes(lay: Layout, n_eff: int):
    """-> ([(class, group index, sweep index)], expectation launches) of ``launch_expectation_t`` for plans of width ``n_eff``."""
    routes, launches = [], 0
    fuse = lay.table and lay.table_n_eff == n_eff
    if fuse:
        routes.append(("D1" if lay.diagonal else "D2", 0, None))
        launches += 1
    elif lay.n_diag:
        assert not (lay.table and lay.table_n_eff == n_eff)  # (the table kernel: the fused epilogue takes this case)
        routes.append(("D5" if lay.table else ("D3" if _staged(lay.groups[0]) else "D4"), 0, None))
        launches += 2
    tiled = bool(lay.sweeps) and lay.tile_n_eff == n_eff
    if tiled:
        for si, sw in enumerate(lay.sweeps):
            routes += [(_tile_class(lay.groups[g]), g, si) for g in sw.groups]
            launches += 2
    generic = list(lay.generic)
    if not tiled:
        generic += [i for i, g in enumerate(lay.groups) if g.xmask and i not in generic]
    for gi in generic:
        if lay.groups[gi].xmask >> n_eff:
            raise RouteError("Pauli term flips a qubit outside the statevector")
        routes.append(("G1" if _staged(lay.groups[gi]) else "G2", gi, None))
        launches += 2
    if not launches:
        routes.append(("E0", None, None))
        launches += 1
    return routes, launches


def device_routes(lay: Layout, n_local: int, index_offset: int):
    """-> ([(class, group index, sweep index)], expectation launches) of ``expectation_state_t`` on a slice of ``n_local``
    qubits at ``index_offset``.  Raises RouteError where the host returns QB_ERR_INVALID."""
    routes, launches = [], 0
    rank_bits = ~((1 << n_local) - 1)
    table = lay.table and lay.table_n_eff == n_local and index_offset == 0
    if table:
        routes.append(("V1", 0, None))
        launches += 2
    done = set()
    if lay.sweeps and n_local >= EXP_TILE_BITS:
        for si, sw in enumerate(lay.sweeps):
            if any(q >= n_local for q in sw.tile_qubits):
                continue
            for g in sw.groups:
                cls = _tile_class(lay.groups[g])
                if cls == "T3" and any(int(v) & rank_bits for v in lay.groups[g].z):
                    cls = "V3"
                routes.append((cls, g, si))
                done.add(g)
            launches += 2
    for gi, g in enumerate(lay.groups):
        if gi in done or (g.xmask == 0 and table):
            continue
        if g.xmask >> n_local:
            raise RouteError("Pauli term flips a qubit outside the local statevector")
        rank_z = any(int(v) & rank_bits for v in g.z)
        if g.xmask == 0:
            cls = "V2" if rank_z else ("D3" if _staged(g) else "D4")
        else:
            cls = "V5" if rank_z else ("G1" if _staged(g) else "G2")
        routes.append((cls, gi, None))
        launches += 2
    if not routes:
        routes.append(("E0", None, None))  # (a memset, no kernel)
    return routes, launches


def features(lay: Layout, routes, device_n_local: int | None = None) -> set:
    """Route classes plus what the kernels branch on inside them."""
    out = {cls for cls, _, _ in routes}
    for cls, gi, si in routes:
        if cls == "T1":
            out.add(f"T1.S{lay.groups[gi].xloc >> 8}")
        if cls in ("T3", "V3"):
            g = lay.groups[gi]
            ny = {bin(g.xmask & int(zz)).count("1") & 1 for zz in g.z}
            out |= {"T3.oddY" if v else "T3.evenY" for v in ny}
            if np.any(g.w.real != 0) and np.any(g.w.imag != 0):
                out.add("T3.complex")
        if cls in ("D3", "D4", "D5", "V2", "G1", "G2", "V5"):
            n_terms = len(lay.groups[gi].z)
            if n_terms in (MAX_STAGED_TERMS, MAX_STAGED_TERMS + 1):
                out.add(f"stage.{n_terms}.{'diag' if lay.groups[gi].xmask == 0 else 'group'}")
    sweeps = {si for _, _, si in routes if si is not None}
    if len(sweeps) > 1:
        out.add("T4.sweeps")
    if any(sum(1 for _, _, s in routes if s == si) > 1 for si in sweeps):
        out.add("T4.groups")
    if lay.sweeps and not sweeps and any(c in ("G1", "G2") for c, _, _ in routes) and device_n_local is None:
        out.add("T5")
    if device_n_local is not None and device_n_local < EXP_TILE_BITS:
        out.add("V4")
    if lay.table_chunks:
        out.add(f"table.chunks{lay.table_chunks}")
    return out


# ----------------------------------------------------------------------------------------------- emulator
def _sign(idx: np.ndarray, z: int) -> np.ndarray:
    return 1.0 - 2.0 * (_popcount(idx & np.uint64(z)) & 1)


def _weights(idx: np.ndarray, g: Group):
    wr, wi = np.zeros(idx.shape), np.zeros(idx.shape)
    for zz, w in zip(g.z, g.w):
        s = _sign(idx, int(zz))
        wr += s * w.real
        wi += s * w.imag
    return wr, wi


def build_table(lay: Layout, n_eff: int, index_offset: int = 0) -> np.ndarray:
    """``fill_diag_table``: E(k) for k < 2^n_eff, chunk after chunk onto the table."""
    k = np.arange(1 << n_eff, dtype=np.uint64) | np.uint64(index_offset)
    table = np.zeros(1 << n_eff)
    for lo in range(0, lay.n_diag, TABLE_TERM_CHUNK):
        e = table.copy()
        for zz, cc in zip(lay.diag_z[lo : lo + TABLE_TERM_CHUNK], lay.diag_c[lo : lo + TABLE_TERM_CHUNK]):
            e += _sign(k, int(zz)) * cc
        table = e
    return table


def _group_value(psi, g: Group, index_offset: int) -> float:
    """``expect_group_kernel``: sum_k Re[psi_k conj(psi_{k^x}) W(k)]."""
    k = np.arange(psi.size, dtype=np.uint64)
    b = psi[(k ^ np.uint64(g.xmask)).astype(np.int64)]
    pr = psi.real * b.real + psi.imag * b.imag
    pi = psi.imag * b.real - psi.real * b.imag
    wr, wi = _weights(k | np.uint64(index_offset), g)
    return float(np.sum(pr * wr - pi * wi))


def _tile_value(psi, lay: Layout, sw: Sweep, n_eff: int, index_offset: int) -> float:
    """``expect_tile_kernel`` for one sweep: element e of a tile sits at global index base | sum_b bit_b(e) << tile_qubits[b]."""
    tq = sw.tile_qubits
    assert len(tq) == EXP_TILE_BITS and all(q < n_eff for q in tq)
    e = np.arange(1 << EXP_TILE_BITS, dtype=np.uint64)
    local = np.zeros_like(e)
    for b, q in enumerate(tq):
        local |= ((e >> np.uint64(b)) & np.uint64(1)) << np.uint64(q)
    outside = [q for q in range(n_eff) if q not in tq]
    t = np.arange(1 << len(outside), dtype=np.uint64)
    base = np.zeros_like(t)
    for i, q in enumerate(outside):
        base |= ((t >> np.uint64(i)) & np.uint64(1)) << np.uint64(q)
    gidx = base[:, None] | local[None, :]
    a = psi[gidx.astype(np.int64)]
    total = 0.0
    for gi in sw.groups:
        g = lay.groups[gi]
        assert int(local[g.xloc]) == g.xmask  # the partner of element 0 is the flipped global index
        b = a[:, (e ^ np.uint64(g.xloc)).astype(np.int64)]
        pr = a.real * b.real + a.imag * b.imag
        if g.trivial:
            total += float(g.w[0].real * np.sum(pr))  # the imaginary parts of a pair cancel
            continue
        pi = a.imag * b.real - a.real * b.imag
        wr, wi = _weights(gidx | np.uint64(index_offset), g)
        total += float(np.sum(pr * wr - pi * wi))
    return total


def emulate(lay: Layout, routes, psi: np.ndarray, n_eff: int, index_offset: int = 0) -> float:
    """The value the route list computes for the state ``psi`` of 2^n_eff amplitudes (one slice of a sharded state)."""
    psi = np.asarray(psi, dtype=np.complex128)
    assert psi.size == 1 << n_eff
    total, swept = 0.0, set()
    for cls, gi, si in routes:
        if cls in ("D1", "D2", "V1"):
            total += float(np.sum((psi.real ** 2 + psi.imag ** 2) * build_table(lay, n_eff)))
        elif si is not None:
            if si not in swept:
                swept.add(si)
                total += _tile_value(psi, lay, lay.sweeps[si], n_eff, index_offset)
        elif cls != "E0":
            total += _group_value(psi, lay.groups[gi], index_offset)
    return total


# ----------------------------------------------------------------------------------------------- reference
def _walsh_hadamard(v: np.ndarray) -> np.ndarray:
    """out[z] = sum_k v[k] (-1)^{pc(k & z)}."""
    n = v.size.bit_length() - 1
    a = v.copy()
    for i in range(n):
        a = a.reshape(-1, 2, 1 << i)
        a = np.concatenate([a[:, 0] + a[:, 1], a[:, 0] - a[:, 1]], axis=1)
    return a.reshape(-1)


def term_values(psi: np.ndarray, x, z) -> np.ndarray:
    """<psi| X^x Z^z |psi> (without i^{#Y}) of every term, each reduced on its own in float64: P|k> = (-1)^{pc(k&z)} |k^x>, so
    <P> = sum_k conj(psi_{k^x}) (-1)^{pc(k&z)} psi_k.  Terms of one x mask share the pair products; many of them are reduced
    all at once by a Walsh-Hadamard transform (n butterfly levels per term instead of a 2^n-term sum)."""
    psi = np.asarray(psi, dtype=np.complex128)
    x = np.asarray(x, dtype=np.uint64)
    z = np.asarray(z, dtype=np.uint64)
    k = np.arange(psi.size, dtype=np.uint64)
    out = np.zeros(len(x), dtype=complex)
    for xm in np.unique(x):
        sel = np.flatnonzero(x == xm)
        pair = np.conj(psi[(k ^ xm).astype(np.int64)]) * psi
        if len(sel) > 8:
            out[sel] = _walsh_hadamard(pair)[z[sel].astype(np.int64)]
        else:
            for t in sel:
                out[t] = np.sum(pair * _sign(k, int(z[t])))
    return out


def reference(psi: np.ndarray, x, z, c) -> float:
    """Re sum_t c_t i^{#Y_t} <X^x Z^z>_t, the terms summed exactly (math.fsum).  ``psi`` may be shorter than 2^n only when no
    term reaches past it (padding qubits stay |0>)."""
    x = np.asarray(x, dtype=np.uint64)
    z = np.asarray(z, dtype=np.uint64)
    c = np.asarray(c, dtype=complex)
    if not len(x):
        return 0.0
    ny = _popcount(x & z) & 3
    vals = term_values(psi, x, z) * c * (1j ** ny)
    return math.fsum(vals.real)


def tolerance(lay: Layout, norm2: float) -> float:
    """Bound on |GPU - reference| of a double-precision reduction of the same amplitudes (tests/test_gpu_expectation_routes.py)."""
    t_max = max([len(g.z) for g in lay.groups] + [lay.n_diag, 1])
    total = float(sum(np.sum(np.abs(g.w)) for g in lay.groups))
    return (2 * (t_max + 8 * len(lay.groups)) + 512) * 2.0 ** -53 * total * max(norm2, 1.0)


# ----------------------------------------------------------------------------------------------- operators
def _op(n, x, z, c):
    from queasars_b200.operators import SparsePauliOp

    return SparsePauliOp._raw(n, [int(v) for v in x], [int(v) for v in z], [complex(v) for v in c])


def _tfim(n, rng):
    x = [0] * (n - 1) + [1 << q for q in range(n)]
    z = [(3 << q) for q in range(n - 1)] + [0] * n
    c = list(rng.normal(size=n - 1)) + list(rng.normal(size=n))
    return x, z, c


def _distinct(rng, count, n, exclude=()):
    assert count + len(exclude) <= 1 << n
    out = rng.choice(1 << n, size=count + len(exclude), replace=False)
    out = [int(v) for v in out if int(v) not in set(exclude)]
    return out[:count]


def operator_family(n: int, seed: int = 0, many_terms: bool | None = None) -> list:
    """-> [(label, operator, build_table)] at width ``n``: every route class, S, staging boundary and table chunk count the width
    allows.  ``many_terms`` (default: 11 <= n <= 14) adds the 2000 / 2001-term groups and 3000 / 3001 / 6001-term diagonals."""
    rng = np.random.default_rng(1000 * seed + n)
    many = (11 <= n <= 14) if many_terms is None else many_terms
    fam = []
    x, z, c = _tfim(n, rng) if n > 1 else ([1], [0], [0.7])
    fam.append(("tfim", _op(n, x, z, c), None))
    # pure X strings: single flips on the tile-local bits 8 / 9 / 10 (each in a sweep of its own when it is the first group) and
    # on the top qubit, multi-bit flips, plus a Z string so that the diagonal part has a few terms
    xs = [1 << q for q in (8, 9, 10, n - 1, 0, n // 2) if q < n]
    xs += [m for m in ((1 << (n - 1)) | 1, 0b1011 << max(0, n - 4), (1 << n) - 1) if m < (1 << n)]
    fam.append(("xstrings", _op(n, xs + [0], [0] * len(xs) + [1 << (n - 1)], list(rng.normal(size=len(xs))) + [0.25]), None))
    for q in (8, 9, 10):  # a lone flip on bit q: one sweep whose element bit q - 8 holds the flipped qubit
        if q < n:
            fam.append((f"x{q}", _op(n, [1 << q], [0], [rng.normal()]), None))
    # X / Y / Z mixes with complex coefficients: several z per x mask (general groups), even and odd #Y
    pool = [m for m in {int(v) for v in rng.integers(1, 1 << n, size=6)} | {1, 1 << (n - 1)}]
    mx, mz = [], []
    for xm in pool:
        for _ in range(3):
            mx.append(xm), mz.append(int(rng.integers(0, 1 << n)))
        mx.append(xm), mz.append(xm)  # all Y on the flipped qubits
        mx.append(xm), mz.append(xm & -xm)  # one Y
    mx += [0, 0, 0]
    mz += [int(v) for v in rng.integers(0, 1 << n, size=3)]
    mc = rng.normal(size=len(mx)) + 1j * rng.normal(size=len(mx))
    fam.append(("mixed", _op(n, mx, mz, mc), None))
    fam.append(("mixed_table", _op(n, mx + [0] * 9, mz + _distinct(rng, 9, n) if n >= 4 else mz + [0] * 9, list(mc) + list(rng.normal(size=9))), True))
    if n >= 12:  # x masks wider than a tile: eight flipped qubits above the four low ones
        wide = 0xFF << 4
        wx = [wide] * 3 + [wide | 1] * 2
        wz = [int(v) for v in rng.integers(0, 1 << n, size=5)]
        wz[1] = wide  # 8 Y
        wz[3] = wide & ~(1 << 4)  # 7 Y and an X
        fam.append(("wide", _op(n, wx + [0], wz + [0], list(rng.normal(size=5) + 1j * rng.normal(size=5)) + [0.5]), None))
    if n >= 4:
        ising_z = [1 << q for q in range(n)] + [(1 << i) | (1 << j) for i in range(n) for j in range(i + 1, n)]
        fam.append(("ising", _op(n, [0] * len(ising_z), ising_z, rng.normal(size=len(ising_z))), True))
        fam.append(("ising_x", _op(n, [0] * len(ising_z) + [1 << (n - 1), 3], ising_z + [0, 2], list(rng.normal(size=len(ising_z))) + [0.3, -0.4]), True))
    fam.append(("identity", _op(n, [0], [0], [1.25]), None))
    fam.append(("empty", _op(n, [], [], []), None))
    if many:
        for count in (MAX_STAGED_TERMS, MAX_STAGED_TERMS + 1):
            zs = _distinct(rng, count, n)
            fam.append((f"diag{count}", _op(n, [0] * count, zs, rng.normal(size=count)), False))
            xm = (0xFF << 4) if n >= 12 else 0b1001100000
            fam.append((f"group{count}", _op(n, [xm] * count, zs, rng.normal(size=count) + 1j * rng.normal(size=count)), None))
        for count in (TABLE_TERM_CHUNK, TABLE_TERM_CHUNK + 1, 2 * TABLE_TERM_CHUNK + 1):
            if count <= 1 << n:
                fam.append((f"table{count}", _op(n, [0] * count, _distinct(rng, count, n), rng.normal(size=count)), True))
    return fam


def device_family(n: int, n_local: int, seed: int = 0) -> list:
    """-> [(label, operator, build_table)] at width ``n`` = ``n_local`` + rank bits: every x mask stays on the local qubits, z
    masks reach the rank bits (general tile groups, the diagonal group, wide generic groups) -- what a sharded state evaluates
    after its global qubits carrying X / Y factors have been swapped local."""
    rng = np.random.default_rng(1000 * seed + 31 * n + n_local)
    rank = [1 << q for q in range(n_local, n)]
    top = (1 << n) - 1
    fam = []
    # general groups in tile sweeps: X / Y on local qubits (bits 8-10 too), Z on rank bits, several z per x
    xs = [m for m in (1 << 8, 1 << (n_local - 1), 0b101, (1 << 9) | 1) if not m >> n_local]
    x, z = [], []
    for xm in xs:
        for r in rank:
            x.append(xm), z.append(r | int(rng.integers(0, 1 << n_local)))
        x.append(xm), z.append(xm | rank[-1])  # Y factors and a rank Z
        x.append(xm), z.append(0)
    if n_local > 9:  # a pure X string beside them (the register-partner path with a rank offset)
        x.append(1 << 9), z.append(0)
    dz = [r | (1 << (n_local - 1)) for r in rank] + [top, 1]
    x += [0] * len(dz)
    z += dz
    fam.append(("rank_z", _op(n, x, z, rng.normal(size=len(x)) + 1j * rng.normal(size=len(x))), None))
    # diagonal with z on rank bits: few terms (on the fly), many terms (a table for the full width, on the fly per slice)
    tz = _distinct(rng, 12, n)
    fam.append(("rank_diag", _op(n, [0] * 12, tz, rng.normal(size=12)), True))
    if n_local >= 12:  # generic group: x wider than a tile on local qubits, z on rank bits
        wide = 0xFF << 4
        fam.append(("rank_wide", _op(n, [wide] * 3, [rank[0], wide | rank[-1], 0], rng.normal(size=3) + 1j * rng.normal(size=3)), None))
    fam.append(("empty", _op(n, [], [], []), None))
    return fam
