"""Exact references for block-product states: amplitudes, Pauli expectations, inverse-CDF draws and exact CVaR of states too wide
for the oracle (27-34 qubits on one GPU: a 33-qubit complex128 state is 128 GiB).  Test infrastructure.

A ``Layout`` partitions the ``n`` qubits into blocks of at most 12 qubits.  Every block gets its own random entangling circuit and
the oracle (``oracle.qiskit_semantics.statevector``) simulates it on the block's qubits alone.  The wide circuit runs all block
circuits interleaved in time; blocks act on disjoint qubits, so they commute and the wide state is the tensor product of the block
states.  Everything below is computed from the blocks:

  amplitude(k)          product of the block amplitudes at k's bits
  <P>                   product of the per-block expectations of P's restriction to the block
  inverse CDF           a descent from bit n-1 to bit 0 in basis-index order: the mass of the set of indices with a fixed prefix
                        is a product of block masses, each a partial sum over the block's indices with that block's prefix bits
  exact CVaR(alpha)     of a diagonal H on a qubit subset S (|S| <= 20): the 2^|S| energies sorted, their masses from the block
                        marginals, the tie groups walked in order, and the stop entry inside the stopping group placed by the
                        descent restricted to the group's S-patterns (the device's order is stable: ascending (E(k), k))

The block qubits interleave bit positions on purpose (``dense_layout``): every block mixes low qubits, the tile-boundary qubits
10-12 and the qubits 29-33 that carry the 2^29 .. 2^33 index bits, and the planner mixes blocks inside sweeps."""
from __future__ import annotations

import functools
import math

import numpy as np

from oracle import qiskit_semantics as oq
from queasars_b200 import expectation as ex

BLOCK_MAX = 12
HIGH = (29, 30, 31, 32, 33)  # the 2^29 .. 2^33 index bits


def _popcount_parity(a: np.ndarray) -> np.ndarray:
    return (np.bitwise_count(np.asarray(a, dtype=np.uint64)) & 1).astype(bool)


class Block:
    """Qubits (ascending; local bit i <-> qubits[i]), the block's circuit on local qubits and its state."""

    def __init__(self, qubits, instr, values: dict):
        self.qubits = tuple(int(q) for q in qubits)
        self.m = len(self.qubits)
        self.local_instr = instr
        names = oq.parameter_names(instr)
        self.psi = oq.statevector(instr, self.m, [values[p] for p in names])
        self.p = self.psi.real**2 + self.psi.imag**2
        self.idx = np.arange(1 << self.m, dtype=np.uint64)

    def local_index(self, k):
        """Global basis indices (uint64 array) -> this block's local indices."""
        k = np.asarray(k, dtype=np.uint64)
        out = np.zeros(k.shape, dtype=np.int64)
        for i, q in enumerate(self.qubits):
            out |= ((k >> np.uint64(q)) & np.uint64(1)).astype(np.int64) << i
        return out

    def local_mask(self, mask: int) -> int:
        return sum(1 << i for i, q in enumerate(self.qubits) if (mask >> q) & 1)

    def pauli(self, x: int, z: int) -> complex:
        """<psi_B| P_B |psi_B> of the restriction (x, z) of a Pauli string, with its i^{#Y} factor."""
        xl, zl = self.local_mask(x), self.local_mask(z)
        ny = bin(xl & zl).count("1")
        sign = np.where(_popcount_parity(self.idx & np.uint64(zl)), -1.0, 1.0)
        partner = self.psi[(self.idx ^ np.uint64(xl)).astype(np.int64)]
        return complex((1j**ny) * np.sum(np.conj(partner) * sign * self.psi))


def levels(w: np.ndarray) -> list:
    """w[..., 2^m] -> L with L[j][..., v] = sum of w over the local indices whose top j bits are v (pairwise from the leaves)."""
    m = w.shape[-1].bit_length() - 1
    out = [None] * (m + 1)
    out[m] = w
    for j in range(m - 1, -1, -1):
        a = out[j + 1]
        out[j] = a.reshape(a.shape[:-1] + (-1, 2)).sum(axis=-1)
    return out


class Layout:
    def __init__(self, n: int, blocks, instr, values: dict):
        self.n, self.blocks, self.instr = n, blocks, instr
        self.names = oq.parameter_names(instr)
        self.values = [values[p] for p in self.names]
        self.block_of = {}
        for bi, b in enumerate(blocks):
            for pos, q in enumerate(b.qubits):
                self.block_of[q] = (bi, pos)
        assert sorted(self.block_of) == list(range(n)), "blocks must partition the qubits"
        self._mass_levels = [levels(b.p) for b in blocks]

    # ------------------------------------------------------------------ amplitudes and Pauli strings
    def amplitudes(self, k) -> np.ndarray:
        k = np.asarray(k, dtype=np.uint64)
        out = np.ones(k.shape, dtype=np.complex128)
        for b in self.blocks:
            out *= b.psi[b.local_index(k)]
        return out

    def probabilities(self, k) -> np.ndarray:
        a = self.amplitudes(k)
        return a.real**2 + a.imag**2

    def max_abs(self) -> float:
        return float(np.prod([np.max(np.abs(b.psi)) for b in self.blocks]))

    def pauli(self, label: str) -> complex:
        """<psi| P |psi> of a Pauli label (right-most char = qubit 0), as ``oq.pauli_expectation``."""
        x, z, _ = oq.pauli_label_to_masks(label)
        out = 1.0 + 0.0j
        for b in self.blocks:
            out *= b.pauli(x, z)
        return out

    def pauli_sum(self, terms) -> float:
        """Re sum_j c_j <P_j> (``oq.estimator_expectation``), terms summed with ``math.fsum``."""
        return math.fsum((complex(c) * self.pauli(lab)).real for lab, c in terms)

    # ------------------------------------------------------------------ inverse CDF in basis-index order
    def _walk(self):
        """(bit, block, level after fixing the bit) from bit n-1 down to 0."""
        for bit in range(self.n - 1, -1, -1):
            bi, pos = self.block_of[bit]
            yield bit, bi, self.blocks[bi].m - pos

    def sample(self, uniforms) -> np.ndarray:
        """searchsorted(cumsum(p) / sum(p), u, side='right') for every uniform: the first k whose inclusive mass exceeds u * total."""
        u = np.asarray(uniforms, dtype=np.float64)
        nb = len(self.blocks)
        v = np.zeros((nb, u.size), dtype=np.int64)
        cur = np.array([[lv[0][0]] * u.size for lv in self._mass_levels])  # mass of each block's part of the current set
        r = u * float(np.prod(cur[:, 0]))
        k = np.zeros(u.size, dtype=np.uint64)
        for bit, bi, j in self._walk():
            left = self._mass_levels[bi][j][2 * v[bi]]
            others = np.prod(np.delete(cur, bi, axis=0), axis=0)
            m0 = left * others
            go_right = r >= m0
            r = np.where(go_right, r - m0, r)
            v[bi] = 2 * v[bi] + go_right
            cur[bi] = np.where(go_right, self._mass_levels[bi][j][v[bi]], left)
            k |= go_right.astype(np.uint64) << np.uint64(bit)
        return k.astype(np.int64)

    def mass_below(self, ks) -> np.ndarray:
        """sum of p_i over i < k for every k (vectorised ``measure_below`` of the plain mass)."""
        k = np.asarray(ks, dtype=np.int64)
        nb = len(self.blocks)
        v = np.zeros((nb, k.size), dtype=np.int64)
        cur = np.array([[lv[0][0]] * k.size for lv in self._mass_levels])
        out = np.zeros(k.size)
        for bit, bi, j in self._walk():
            one = (k >> bit) & 1
            left = self._mass_levels[bi][j][2 * v[bi]]
            out += np.where(one == 1, left * np.prod(np.delete(cur, bi, axis=0), axis=0), 0.0)
            v[bi] = 2 * v[bi] + one
            cur[bi] = self._mass_levels[bi][j][v[bi]]
        return out

    def _tables(self, weights):
        """weights: per block (array [U_B, 2^m_B] of weights over local indices, index array [T] into it) -> level tables."""
        return [(levels(w * b.p), np.asarray(ix, dtype=np.int64)) for b, (w, ix) in zip(self.blocks, weights)]

    def descend(self, target: float, weights=None, coeffs=None, side: str = "left"):
        """Inverse CDF of the measure mu(A) = sum_t coeffs[t] prod_B sum_{k in A} w_{B,t}(k_B) p_B(k_B) in basis-index order.
        side 'left': the first k with mu([0, k]) >= target; 'right': the first k with mu([0, k]) > target.
        -> (k, mu([0, k)), mu({k})).  Without weights mu is the plain probability mass."""
        if weights is None:
            weights = [(np.ones((1, 1 << b.m)), [0]) for b in self.blocks]
            coeffs = [1.0]
        tabs = self._tables(weights)
        coeffs = np.asarray(coeffs, dtype=np.float64)
        v = [0] * len(tabs)
        cur = [lv[0][:, 0][ix] for lv, ix in tabs]  # per block and term: weight of the block's part of the current set
        r, before, k = float(target), 0.0, 0
        for bit, bi, j in self._walk():
            lv, ix = tabs[bi]
            left = lv[j][:, 2 * v[bi]][ix]
            prod = coeffs * left
            for bj, c in enumerate(cur):
                if bj != bi:
                    prod = prod * c
            m0 = math.fsum(prod)
            if (r <= m0) if side == "left" else (r < m0):
                v[bi] = 2 * v[bi]
                cur[bi] = left
            else:
                r -= m0
                before += m0
                v[bi] = 2 * v[bi] + 1
                cur[bi] = lv[j][:, v[bi]][ix]
                k |= 1 << bit
        here = coeffs.copy()
        for c in cur:
            here = here * c
        return k, before, math.fsum(here)

    def measure_below(self, k: int, weights=None, coeffs=None) -> float:
        """mu({i < k}) of the measure of ``descend``: the union of the left siblings of k's path."""
        if weights is None:
            weights = [(np.ones((1, 1 << b.m)), [0]) for b in self.blocks]
            coeffs = [1.0]
        tabs = self._tables(weights)
        coeffs = np.asarray(coeffs, dtype=np.float64)
        v = [0] * len(tabs)
        cur = [lv[0][:, 0][ix] for lv, ix in tabs]
        parts = []
        for bit, bi, j in self._walk():
            lv, ix = tabs[bi]
            one = (k >> bit) & 1
            if one:
                prod = coeffs * lv[j][:, 2 * v[bi]][ix]
                for bj, c in enumerate(cur):
                    if bj != bi:
                        prod = prod * c
                parts.append(math.fsum(prod))
            v[bi] = 2 * v[bi] + one
            cur[bi] = lv[j][:, v[bi]][ix]
        return math.fsum(parts)

    # ------------------------------------------------------------------ diagonal Hamiltonians on a qubit subset
    def _sign_weights(self, z_masks):
        """Per block: the distinct sign patterns (-1)^{popcount(k_B & z_B)} of the terms, and each term's row."""
        out = []
        for b in self.blocks:
            rows, ix = {}, []
            for z in z_masks:
                zl = b.local_mask(int(z))
                ix.append(rows.setdefault(zl, len(rows)))
            w = np.array([np.where(_popcount_parity(b.idx & np.uint64(zl)), -1.0, 1.0) for zl in rows])
            out.append((w, ix))
        return out

    def _pattern_weights(self, S, patterns):
        """Per block: indicator rows of the block's S-bits equal to each pattern's, and each pattern's row."""
        out = []
        for b in self.blocks:
            bits = [(i, S.index(q)) for i, q in enumerate(b.qubits) if q in S]
            local = np.zeros(len(patterns), dtype=np.int64)
            for i, s in bits:
                local |= ((np.asarray(patterns) >> s) & 1) << i
            keys, ix = np.unique(local, return_inverse=True)
            mask = sum(1 << i for i, _ in bits)
            w = np.array([((b.idx.astype(np.int64) & mask) == kk).astype(np.float64) for kk in keys])
            out.append((w, ix.reshape(-1)))
        return out

    def pattern_masses(self, S) -> np.ndarray:
        """P(S-bits = s) for every pattern s (bit i of s <-> qubit S[i]), from the block marginals."""
        out = np.ones(1, dtype=np.float64)
        width = 0
        for b in self.blocks:
            bits = [(i, S.index(q)) for i, q in enumerate(b.qubits) if q in S]
            if not bits:
                continue
            marg = np.zeros(1 << len(bits))
            sub = np.zeros(1 << b.m, dtype=np.int64)
            for j, (i, _) in enumerate(bits):
                sub |= ((b.idx.astype(np.int64) >> i) & 1) << j
            np.add.at(marg, sub, b.p)
            out = np.outer(marg, out).reshape(-1)  # new block's bits above the ones collected so far
            width += len(bits)
        order = [s for b in self.blocks for _, s in [(i, S.index(q)) for i, q in enumerate(b.qubits) if q in S]]
        # collected index: bit j <-> S-position order[j]; permute to bit i <-> S[i]
        col = np.arange(1 << width)
        pat = np.zeros(1 << width, dtype=np.int64)
        for j, s in enumerate(order):
            pat |= ((col >> j) & 1) << s
        masses = np.empty(1 << width)
        masses[pat] = out
        return masses

    @staticmethod
    def pattern_energies(S, z_masks, coeffs) -> np.ndarray:
        """E of every S-pattern, summed term after term from 0.0 as ``diag_table_kernel`` does (the same doubles, the same ties)."""
        pats = np.arange(1 << len(S), dtype=np.uint64)
        e = np.zeros(pats.size)
        for z, c in zip(z_masks, coeffs):
            zl = sum(1 << i for i, q in enumerate(S) if (int(z) >> q) & 1)
            e = e + np.where(_popcount_parity(pats & np.uint64(zl)), -float(c), float(c))
        return e

    def energy(self, k: int, z_masks, coeffs) -> float:
        e = 0.0
        for z, c in zip(z_masks, coeffs):
            e += -float(c) if bin(k & int(z)).count("1") & 1 else float(c)
        return e

    def cvar(self, S, z_masks, coeffs, alpha: float, bound_shift: float = 0.0) -> float:
        """expectation.lower_tail_expectation_arrays(|psi|^2, E, alpha) over all 2^n basis states for E(k) = sum_t c_t
        (-1)^{popcount(k & z_t)}, every z_t inside S.  ``bound_shift`` moves the stop bound alpha - isclose tolerance (to find
        the stop entries a summation order within that distance could pick)."""
        return self.cvar_stop(S, z_masks, coeffs, alpha, bound_shift)[0]

    def cvar_stop(self, S, z_masks, coeffs, alpha: float, bound_shift: float = 0.0):
        """-> (CVaR value, basis index of the entry the greedy fill stops at; None when the whole mass is below the bound)."""
        S = sorted(int(q) for q in S)
        assert all(int(z) & ~sum(1 << q for q in S) == 0 for z in z_masks)
        bound = alpha - (ex._ATOL + ex._RTOL * abs(alpha)) + bound_shift
        if ex._close(alpha, 1):  # greedy fill in basis order
            k, before, pk = self.descend(bound)
            acc = self.measure_below(k, self._sign_weights(z_masks), coeffs)
            return (acc + min(alpha - before, pk) * self.energy(k, z_masks, coeffs)) / alpha, k
        E = self.pattern_energies(S, z_masks, coeffs)
        P = self.pattern_masses(S)
        order = np.argsort(E, kind="stable")
        Es, Ps = E[order], P[order]
        starts = np.flatnonzero(np.concatenate(([True], Es[1:] != Es[:-1])))
        ends = np.concatenate((starts[1:], [Es.size]))
        cum, acc = 0.0, []
        for lo, hi in zip(starts, ends):
            g = math.fsum(Ps[lo:hi])
            e = float(Es[lo])
            if cum + g >= bound:
                members = order[lo:hi]
                k, within, pk = self.descend(bound - cum, self._pattern_weights(S, members), np.ones(members.size))
                take = within + min(alpha - (cum + within), pk)
                return (math.fsum(acc) + take * e) / alpha, k
            cum += g
            acc.append(g * e)
        return math.fsum(acc) / alpha, None


# ------------------------------------------------------------------------------------------------ layouts
def _block_circuit(qubits, high, rng, depth, tag):
    """Random entangling circuit on local qubits 0..m-1 (qubits[i] global): u on every qubit first (so the product-state start
    folds every qubit), then layers of u / ry / rz / cx / cu3 / rzz / crx, with X / Y gates and controls on the high qubits."""
    m = len(qubits)
    hi = [i for i, q in enumerate(qubits) if q in high]
    names = iter(f"{tag}_{i:03d}" for i in range(10**6))
    vals = {}

    def prm():
        name = next(names)
        vals[name] = float(rng.uniform(-math.pi, math.pi))
        return name

    def angles(k):
        return tuple(float(a) for a in rng.uniform(-math.pi, math.pi, k))

    instr = [("u", (i,), angles(3)) for i in range(m)]
    for _ in range(depth):
        for i in rng.permutation(m):
            i = int(i)
            r = rng.random()
            if r < 0.3:
                instr.append(("ry", (i,), (prm(),)))
            elif r < 0.5:
                instr.append(("rz", (i,), (prm(),)))
            elif r < 0.6:
                instr.append(("u", (i,), angles(3)))
        pairs = rng.permutation(m)
        for a, b in zip(pairs[0::2], pairs[1::2]):
            a, b = int(a), int(b)
            kind = rng.choice(["cx", "cu3", "rzz", "crx"])
            if kind == "cx":
                instr.append(("cx", (a, b), ()))
            elif kind == "cu3":
                instr.append(("cu3", (a, b), angles(3)))
            else:
                instr.append((str(kind), (a, b), (prm(),)))
        for i in hi:  # X / Y on the high qubits, and gates they control
            instr.append((("x", "y")[int(rng.integers(2))], (i,), ()))
            t = int(rng.choice([j for j in range(m) if j != i]))
            name = ("cx", "crx", "cu3")[int(rng.integers(3))]
            instr.append((name, (i, t), () if name == "cx" else ((prm(),) if name == "crx" else angles(3))))
            if len(hi) > 1:
                o = int(rng.choice([j for j in hi if j != i]))
                instr.append(("rzz", (i, o), (prm(),)))
    # a closing layer: dense gates on the other qubits fill a tile, then diagonals and controls on the high qubits, which the
    # planner applies from outside that tile
    instr += [("u", (j,), angles(3)) for j in range(m) if j not in hi]
    for i in hi:
        lo = int(rng.choice([j for j in range(m) if j not in hi] or [j for j in range(m) if j != i]))
        instr += [("rzz", (lo, i), (prm(),)), ("crz", (lo, i), (prm(),)), ("cx", (i, lo), ())]
    instr += [("rzz", (a, b), (prm(),)) for a, b in zip(hi, hi[1:])]
    return instr, vals


def _interleave(per_block, rng):
    """All block circuits merged in time, the next instruction taken from a random block that still has some."""
    pos = [0] * len(per_block)
    out = []
    while True:
        live = [i for i, ins in enumerate(per_block) if pos[i] < len(ins)]
        if not live:
            return out
        i = int(rng.choice(live))
        out.append(per_block[i][pos[i]])
        pos[i] += 1


def make_layout(n: int, groups, seed: int, depth: int = 3, high=HIGH, idle=()) -> Layout:
    """Blocks ``groups`` (lists of global qubits) with random circuits; qubits in ``idle`` get no gates (stay |0>)."""
    rng = np.random.default_rng(seed)
    blocks, per_block, values = [], [], {}
    for gi, qs in enumerate(groups):
        qs = sorted(qs)
        assert len(qs) <= BLOCK_MAX
        if set(qs) <= set(idle):
            local, vals = [], {}
        else:
            local, vals = _block_circuit(qs, high, rng, depth, f"b{gi}")
        values.update(vals)
        blocks.append(Block(qs, local, vals))
        per_block.append([(name, tuple(qs[i] for i in qubits), params) for name, qubits, params in local])
    return Layout(n, blocks, _interleave(per_block, rng), values)


def dense_groups(n: int, block_max: int = BLOCK_MAX, rotate: int = 0):
    """Qubits dealt round robin over ceil(n / block_max) blocks: each block gets low qubits, one of 10-12 and some of 29-33."""
    nb = -(-n // block_max)
    return [[q for q in range(n) if (q + rotate) % nb == b] for b in range(nb)]


@functools.lru_cache(maxsize=None)
def dense_layout(n: int, seed: int = 0, depth: int = 3, block_max: int = BLOCK_MAX) -> Layout:
    return make_layout(n, dense_groups(n, block_max, seed), 1000 * n + seed, depth, high=set(high_qubits(n)))


def sparse_active(n: int):
    """Qubits of the sparse layout: 0, 1 and four high ones (29-33 where they exist, else the top four)."""
    high = [q for q in HIGH if 1 < q < n][-4:]
    if len(high) < 4:
        high = list(range(n - 4, n))
    return sorted({0, 1, *high})


@functools.lru_cache(maxsize=None)
def sparse_layout(n: int, seed: int = 0) -> Layout:
    """An entangled state on ``sparse_active(n)``, every other qubit |0>: at most 64 indices carry mass."""
    active = sparse_active(n)
    rest = [q for q in range(n) if q not in active]
    groups = [active] + [rest[i : i + BLOCK_MAX] for i in range(0, len(rest), BLOCK_MAX)]
    return make_layout(n, groups, 7000 + n + seed, depth=4, high=set(active), idle=rest)


def sparse_support(lay: Layout) -> np.ndarray:
    """The indices that can carry mass (ascending)."""
    act = lay.blocks[0].qubits
    ks = np.zeros(1 << len(act), dtype=np.int64)
    for i, q in enumerate(act):
        ks |= ((np.arange(ks.size) >> i) & 1) << q
    return np.sort(ks)


# ------------------------------------------------------------------------------------------------ operators
def label(n: int, ops: dict) -> str:
    """{qubit: 'X' | 'Y' | 'Z'} -> Pauli label (right-most char = qubit 0)."""
    chars = ["I"] * n
    for q, c in ops.items():
        chars[n - 1 - q] = c
    return "".join(chars)


def high_qubits(n: int):
    """29-33 where at least three of them exist, else the top five qubits."""
    hq = [q for q in HIGH if q < n]
    return hq if len(hq) >= 3 else list(range(n - 5, n))


def tfim_terms(n: int, seed: int = 0):
    """ZZ on neighbours, X on every qubit, Y and XX / YY / XZY strings on the high qubits, and one X string over 12 qubits that
    does not fit a 2^11-amplitude tile (generic kernel)."""
    rng = np.random.default_rng(seed + n)
    hq = high_qubits(n)
    c = lambda: float(rng.uniform(-1, 1))
    terms = [(label(n, {q: "Z", q + 1: "Z"}), c()) for q in range(n - 1)]
    terms += [(label(n, {q: "X"}), c()) for q in range(n)]
    terms += [(label(n, {q: "Y"}), c()) for q in hq]
    terms += [(label(n, {hq[0]: "X", hq[-1]: "X"}), c()), (label(n, {hq[1]: "Y", hq[2]: "Y"}), c())]
    terms += [(label(n, {hq[0]: "X", hq[2]: "Z", hq[-1]: "Y", 11: "Z"}), c())]
    terms += [(label(n, {q: "X" for q in list(range(4, 11)) + hq}), c())]
    return terms


def ising_subset(n: int):
    """S: at most 20 qubits mixing low, tile-boundary and the high qubits."""
    hq = high_qubits(n)
    S = sorted({q for q in (0, 1, 2, 5, 7, 10, 11, 12, 16, 20, 24, n - 1) if q < n} | set(hq))
    assert len(S) <= 20
    return S


def ising_on(n: int, S, seed: int = 0):
    """Z and ZZ terms on S with coefficients in halves (many exact ties): (z_masks, coeffs, labels-and-coefficients)."""
    rng = np.random.default_rng(seed + 31 * n)
    vals = [-1.5, -1.0, -0.5, 0.5, 1.0, 1.5]
    z, c = [], []
    for q in S:
        z.append(1 << q), c.append(float(rng.choice(vals)))
    for a, b in zip(S, S[1:] + S[:1]):
        z.append((1 << a) | (1 << b)), c.append(float(rng.choice(vals)))
    for _ in range(6):
        a, b = (int(v) for v in rng.choice(S, 2, replace=False))
        m = (1 << a) | (1 << b)
        if m not in z:
            z.append(m), c.append(float(rng.choice(vals)))
    terms = [(label(n, {q: "Z" for q in S if (zz >> q) & 1}), cc) for zz, cc in zip(z, c)]
    return z, c, terms


def observable_sets(n: int, seed: int = 0):
    """Eight observables drawn from one pool of strings on the high qubits (shared strings, different coefficients)."""
    rng = np.random.default_rng(seed + 5 * n)
    hq = high_qubits(n)
    pool = [label(n, {q: p}) for q in hq for p in "XYZ"]
    pool += [label(n, {a: p, b: p}) for a, b in zip(hq, hq[1:]) for p in "XYZ"]
    pool += [label(n, {hq[0]: "X", hq[1]: "Y", hq[-1]: "Z"}), label(n, {0: "Z", hq[2]: "X", 11: "Y"})]
    pool += [label(n, {q: "X" for q in list(range(4, 11)) + hq})]
    obs = []
    for _ in range(8):
        pick = rng.choice(len(pool), size=int(rng.integers(4, 9)), replace=False)
        obs.append([(pool[int(i)], float(rng.uniform(-1, 1))) for i in pick])
    return obs
