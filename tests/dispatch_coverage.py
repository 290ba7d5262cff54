"""Which body of the sweep kernel every op of an encoded plan runs, and circuits that reach all of them.  Test infrastructure.

``classify`` restates the staging loop of ``sweep_kernel`` (csrc/qb_kernels.cuh: the loop that builds ``s_word0`` / ``s_ext``)
and the branch order of ``apply_op`` for one pass op.  The body classes are

  dense  {plain, real00, phase} x control {none, reg, thread, ext}   (plain: variant 48 + b, only uncontrolled)
  diag   target {reg, thread, ext} x control {none, reg, thread, ext}

with the register target bit B (dense ops, register-target diagonals), the register control bit CB (register-controlled dense
ops) and, for register-controlled diagonals, the branch of the generic body (``treg`` or ``diag_select``).

``circuit_family`` builds seeded random circuits over the whole gate set the front end lowers, with parameters and affine
expressions, plus directed circuits that reach the rare classes (diagonals with target and control outside the tile, every
register pair of controlled dense ops with and without a global phase, zero and partial product starts).  All of them are
oracle instruction lists (``oracle.qiskit_semantics``)."""
from __future__ import annotations

import collections
import math

import numpy as np

from queasars_b200 import engine as qe
from queasars_b200 import gate_list as gl
from queasars_b200.schedule import K_EXT, K_NONE, K_REG, K_THREAD
from tests.test_frontend_planner import build_circuit

KIND_NAME = {K_NONE: "none", K_REG: "reg", K_THREAD: "thread", K_EXT: "ext"}
CTRLS = ("none", "reg", "thread", "ext")
DENSE_CLASSES = [("dense", "plain", "none")] + [("dense", form, c) for form in ("real00", "phase") for c in CTRLS]
DIAG_CLASSES = [("diag", t, c) for t in ("reg", "thread", "ext") for c in CTRLS]
ALL_CLASSES = DENSE_CLASSES + DIAG_CLASSES  # 21 bodies

# After phase deferral (drop_final_phases=True) every uncontrolled dense gate has phi == 0, so it runs the plain body: the
# uncontrolled real-top-left class exists only in plans that keep the circuit as written.
UNREACHABLE_WHEN_DROPPED = {("dense", "real00", "none")}


def expected_classes(drop_final_phases: bool) -> set:
    return set(ALL_CLASSES) - (UNREACHABLE_WHEN_DROPPED if drop_final_phases else set())


def _zero(ang, j) -> bool:
    return ang["slot"][j] < 0 and ang["slot2"][j] < 0 and ang["const"][j] == 0.0


def classify(po, ang) -> dict:
    """Body class of one ``qb_pass_op`` record (``po``) with its angle record (``ang``), as the kernel stages it."""
    ck, tk = int(po["ctrl_kind"]), int(po["tgt_kind"])
    ctrl = KIND_NAME[ck]
    out = {"B": None, "CB": None, "branch": None, "tgt": KIND_NAME[tk], "ctrl": ctrl}
    if int(po["kind"]) == gl.DENSE:
        assert tk == K_REG
        out["B"] = int(po["tgt_pos"])
        if ck == K_REG:
            out["CB"] = int(po["ctrl_pos"])
        if _zero(ang, 0):  # gamma == 0: real top-left entry
            form = "plain" if (ck == K_NONE and _zero(ang, 2)) else "real00"  # phi == 0 too, and no control of any kind
        else:
            form = "phase"
        out["cls"] = ("dense", form, ctrl)
    else:
        out["cls"] = ("diag", KIND_NAME[tk], ctrl)
        if tk == K_REG:
            out["B"] = int(po["tgt_pos"])
        if ck == K_REG:
            out["CB"] = int(po["ctrl_pos"])
            out["branch"] = "treg" if tk == K_REG else "diag_select"
    return out


# ----------------------------------------------------------------------------------------------- dispatch words
def dispatch_variant(po, ang, reg_bits: int) -> int:
    """The low six bits of the dispatch word the kernel stages for ``po`` (v_dense / v_ctrl / v_diag_* of qb_kernels.cuh)."""
    R = reg_bits
    c = classify(po, ang)
    kind, a, b = c["cls"]
    if kind == "dense":
        B, CB = c["B"], c["CB"]
        v = B if CB is None else R + B * (R - 1) + (CB if CB < B else CB - 1)
        if a in ("plain", "real00"):
            v |= 32
        if a == "plain":
            v |= 16
        return v
    if c["CB"] is not None:
        return R * R + 1 + R
    if a == "reg":
        return R * R + 1 + c["B"]
    return R * R


def decode_variant(v: int, reg_bits: int) -> tuple:
    """The body ``apply_op`` (and the op loop's plain fast path) selects for variant ``v``, in the kernel's branch order."""
    R = reg_bits
    if (v ^ 48) < R:
        return ("dense", "plain", v & 3, None)
    if (v ^ 32) < R:
        return ("dense", "real00", v & 3, None)
    if v & 32:
        c = (v & 31) - R
        B, k = divmod(c, R - 1)
        return ("dense", "real00", B, k if k < B else k + 1) if B < R else ("bad", v)
    if v < R:
        return ("dense", "phase", v, None)
    if v < R * R:
        B, k = divmod(v - R, R - 1)
        return ("dense", "phase", B, k if k < B else k + 1)
    if v == R * R:
        return ("diag", "out", None, None)
    if v < R * R + 1 + R:
        return ("diag", "reg", v - (R * R + 1), None)
    if v == R * R + 1 + R:
        return ("diag", "gen", None, None)
    return ("bad", v)


# ----------------------------------------------------------------------------------------------- plans
def plan_for(gates: gl.GateList, tile_bits: int, reg_bits: int, drop_final_phases: bool, from_zero_state: bool = True):
    """The encoded program the engine uploads for ``gates`` (same cached object: ``engine.encoded_plan``)."""
    g = qe.rewritten(gates, drop_final_phases)
    return g, qe.encoded_plan(g, tile_bits, reg_bits, from_zero_state)[3]


def plan_records(encoded):
    sweeps, passes, pass_ops, angles, init_ops = encoded
    n = sum(int(p["op_end"] - p["op_begin"]) for p in passes)
    for po in pass_ops[:n]:
        yield po, angles[int(po["op_index"])]


class Coverage:
    """Counts of body classes, register bits and branches over a set of encoded plans."""

    def __init__(self, reg_bits: int):
        self.reg_bits = reg_bits
        self.classes = collections.Counter()
        self.dense_bits = collections.Counter()  # (form, B) of uncontrolled dense ops
        self.diag_bits = collections.Counter()  # B of uncontrolled register-target diagonals
        self.ctrl_pairs = collections.Counter()  # (form, B, CB) of register-controlled dense ops
        self.branches = collections.Counter()  # branch of register-controlled diagonals
        self.starts = collections.Counter()  # zero / full / partial product start

    def add(self, encoded):
        init = encoded[4]
        folded = int(np.count_nonzero(init >= 0))
        self.starts["zero" if folded == 0 else ("partial" if folded < len(init) else "full")] += 1
        for po, ang in plan_records(encoded):
            c = classify(po, ang)
            self.classes[c["cls"]] += 1
            kind, a, ctrl = c["cls"]
            if kind == "dense" and ctrl == "none":
                self.dense_bits[(a, c["B"])] += 1
            elif kind == "dense" and ctrl == "reg":
                self.ctrl_pairs[(a, c["B"], c["CB"])] += 1
            elif kind == "diag" and a == "reg" and ctrl == "none":
                self.diag_bits[c["B"]] += 1
            if c["branch"]:
                self.branches[c["branch"]] += 1
        return self

    def missing(self, drop_final_phases: bool) -> list:
        """Everything the kernel dispatches on that these plans did not reach."""
        R = self.reg_bits
        out = [("class",) + c for c in sorted(expected_classes(drop_final_phases)) if not self.classes[c]]
        forms = ("plain", "phase") if drop_final_phases else ("plain", "real00", "phase")
        out += [("dense bit", f, b) for f in forms for b in range(R) if not self.dense_bits[(f, b)]]
        out += [("diag bit", b) for b in range(R) if not self.diag_bits[b]]
        out += [("ctrl pair", f, b, cb) for f in ("real00", "phase") for b in range(R) for cb in range(R) if b != cb and not self.ctrl_pairs[(f, b, cb)]]
        out += [("branch", br) for br in ("treg", "diag_select") if not self.branches[br]]
        return out

    def report(self) -> str:
        lines = [f"  {'/'.join(c):22s} {self.classes[c]}" for c in ALL_CLASSES]
        lines.append(f"  branches {dict(self.branches)}  starts {dict(self.starts)}")
        lines.append(f"  ctrl pairs {len(self.ctrl_pairs)}  dense bits {len(self.dense_bits)}  diag bits {len(self.diag_bits)}")
        return "\n".join(lines)


# ----------------------------------------------------------------------------------------------- circuits
ONE_FIXED = ("x", "y", "z", "h", "s", "sdg", "t", "tdg", "sx", "sxdg")
ONE_PARAM = {"rx": 1, "ry": 1, "rz": 1, "p": 1, "u2": 2, "u": 3}
TWO_FIXED = ("cx", "cy", "cz", "ch", "swap", "ecr")
TWO_PARAM = {"cp": 1, "crz": 1, "crx": 1, "cry": 1, "rzz": 1, "rxx": 1, "rzx": 1, "cu3": 3, "cu": 4}


class _Params:
    """Parameter names p00, p01, ... (name-sorted = slot order) and a value source: a float, a bare name or (coeff, name, const)."""

    def __init__(self, rng, n_names: int):
        self.rng, self.names = rng, [f"p{i:02d}" for i in range(n_names)]

    def draw(self, nonzero: bool = False):
        r = self.rng.random()
        if r < 0.35:
            return str(self.rng.choice(self.names))
        if r < 0.7:
            return (float(self.rng.choice([-2.0, -0.5, 0.75, 1.5])), str(self.rng.choice(self.names)), float(self.rng.uniform(-1, 1)))
        v = float(self.rng.uniform(-math.pi, math.pi))
        return v if (v != 0.0 or not nonzero) else 0.3


def random_circuit(n: int, n_gates: int, seed: int, n_names: int = 6) -> list:
    """Seeded random circuit over the full lowered gate set (every qubit pair, parameters and affine expressions); ``cu`` with a
    non-zero global phase is weighted up so that controlled bodies with a phase occur often."""
    rng = np.random.default_rng(seed)
    prm = _Params(rng, n_names)
    instr = []
    for _ in range(n_gates):
        r = rng.random()
        if r < 0.35:
            q = int(rng.integers(n))
            if rng.random() < 0.3:
                instr.append((str(rng.choice(ONE_FIXED)), (q,), ()))
            else:
                name = str(rng.choice(list(ONE_PARAM)))
                instr.append((name, (q,), tuple(prm.draw() for _ in range(ONE_PARAM[name]))))
        else:
            a, b = (int(v) for v in rng.choice(n, size=2, replace=False))
            if r < 0.5:
                instr.append((str(rng.choice(TWO_FIXED)), (a, b), ()))
            elif r < 0.62:
                instr.append(("cu", (a, b), tuple(prm.draw() for _ in range(3)) + (prm.draw(nonzero=True),)))
            else:
                name = str(rng.choice(list(TWO_PARAM)))
                instr.append((name, (a, b), tuple(prm.draw() for _ in range(TWO_PARAM[name]))))
    return instr


def register_cluster_circuit(n: int, qubits, seed: int) -> list:
    """Every ordered (target, control) pair of ``qubits`` as cu3 (real top-left) and cu (global phase) right behind dense gates
    on all of them: one pass holds the cluster in registers, so every (B, CB) register pair is dispatched.  Also register-target
    diagonals on each of them and register-controlled diagonals with a register or a thread-bit target."""
    rng = np.random.default_rng(seed)
    prm = _Params(rng, 4)
    qs = list(qubits)
    others = [q for q in range(n) if q not in qs]
    instr = [("h", (q,), ()) for q in range(n)]  # every qubit leaves |0> (product start), nothing below is dropped
    instr += [("u", (q,), (prm.draw(), prm.draw(), prm.draw())) for q in qs]  # real00 / plain after deferral, bits 0..R-1
    for t in qs:
        for c in qs:
            if c != t:
                instr.append(("cu3", (c, t), (prm.draw(), prm.draw(), prm.draw())))
    for q in qs:
        instr.append(("rz", (q,), (prm.draw(),)))
        instr.append(("sx", (q,), ()))  # uncontrolled dense with a global phase
    for t in qs:
        for c in qs:
            if c != t:
                instr.append(("cu", (c, t), (prm.draw(), prm.draw(), prm.draw(), prm.draw(nonzero=True))))
    for q in qs:
        instr.append(("ry", (q,), (prm.draw(),)))  # plain: real first column
    for i, t in enumerate(qs):
        instr.append(("cp", (qs[i - 1], t), (prm.draw(),)))  # register control, register target (treg)
        instr.append(("crz", (t, others[i % len(others)]), (prm.draw(),)))  # register control, target elsewhere (diag_select)
    return instr


def outside_tile_circuit(n: int, tile_bits: int, seed: int) -> list:
    """Dense gates on qubits 0 .. tile_bits-1 fill one sweep's tile; diagonals and controls on the qubits above it are then
    external operands of that sweep: diagonal target and control both outside the tile, each of them alone outside, and dense
    gates (real top-left and with a phase) controlled from outside."""
    assert tile_bits >= 11 and n >= tile_bits + 3  # (the operands below name qubits up to 10)
    rng = np.random.default_rng(seed)
    prm = _Params(rng, 4)
    K = tile_bits
    hi = list(range(K, n))
    instr = [("ry", (q,), (prm.draw(),)) for q in range(n)]  # product start: every qubit folds
    instr += [("u", (q,), (prm.draw(), prm.draw(), prm.draw())) for q in range(K - 1)]  # fill the tile of the next sweep
    # qubit K-1 joins the tile with a dense gate further down; diagonals before it find it on a thread bit of the first pass
    instr += [("cp", (hi[1], K - 1), (prm.draw(),)), ("cz", (K - 1, hi[0]), ()), ("crz", (hi[2], K - 1), (prm.draw(),))]
    instr += [("u", (K - 1,), (prm.draw(), prm.draw(), prm.draw()))]
    instr += [
        ("cz", (hi[0], hi[1]), ()),
        ("cp", (hi[1], hi[2]), (prm.draw(),)),
        ("crz", (hi[2], hi[0]), (prm.draw(),)),
        ("rzz", (hi[0], hi[2]), (prm.draw(),)),
        ("rz", (hi[1],), (prm.draw(),)),
        ("t", (hi[2],), ()),
        ("cz", (1, hi[0]), ()),  # control in the tile, target outside
        ("cp", (hi[1], 2), (prm.draw(),)),  # control outside, target in the tile
        ("crz", (hi[2], 9), (prm.draw(),)),
        ("cu3", (hi[0], 5), (prm.draw(), prm.draw(), prm.draw())),
        ("cx", (hi[1], 6), ()),
        ("cu", (hi[2], 7), (prm.draw(), prm.draw(), prm.draw(), prm.draw(nonzero=True))),
        ("cy", (hi[0], 8), ()),
        ("cp", (3, 4), (prm.draw(),)),
        ("cz", (0, 10), ()),
    ]
    instr += [("u", (q,), (prm.draw(), prm.draw(), prm.draw())) for q in range(K)]
    instr += [("rzz", (hi[1], hi[2]), (prm.draw(),)), ("cp", (hi[0], hi[1]), (prm.draw(),))]
    return instr


def partial_start_circuit(n: int, seed: int) -> list:
    """Only some qubits fold into the product start: the others are first reached by a controlled gate, or their first gate
    is controlled by a still untouched qubit (dropped)."""
    rng = np.random.default_rng(seed)
    prm = _Params(rng, 3)
    instr = [("rx", (q,), (prm.draw(),)) for q in range(0, n, 2)]
    instr += [("cx", (q, q + 1), ()) for q in range(0, n - 1, 2)]  # odd qubits: first reached by a controlled gate
    instr += [("cz", (n - 1, 0), ())] if n % 2 == 0 else []
    return instr + random_circuit(n, 40, seed + 1, 3)


def zero_start_circuit(n: int, seed: int) -> list:
    """Opens with controlled gates and diagonals on every qubit; meant for plans compiled for an existing state
    (``from_zero_state=False``), which the kernel starts from |0...0> without a product factor."""
    rng = np.random.default_rng(seed)
    prm = _Params(rng, 3)
    instr = [("cz", (q, (q + 1) % n), ()) for q in range(n)]
    instr += [("cx", ((q + 3) % n, q), ()) for q in range(n)]
    instr += [("rz", (q,), (prm.draw(),)) for q in range(n)]
    return instr + random_circuit(n, 40, seed + 1, 3)


def circuit_family(n: int, tile_bits: int, seed: int = 0, n_random: int = 2, n_gates: int = 120) -> list:
    """-> list of (label, instructions) at width ``n``: random circuits plus the directed ones that fit the width."""
    fam = [(f"random{i}", random_circuit(n, n_gates, seed * 1000 + 17 * n + i)) for i in range(n_random)]
    cluster = [q for q in (5, 6, 8, 9) if q < n]
    if len(cluster) == 4:
        fam.append(("cluster4", register_cluster_circuit(n, cluster, seed + 31)))
        fam.append(("cluster3", register_cluster_circuit(n, [4, 7, 10 if n > 10 else 3], seed + 37)))
    if n >= tile_bits + 3:
        fam.append(("outside", outside_tile_circuit(n, tile_bits, seed + 41)))
    fam.append(("partial", partial_start_circuit(n, seed + 43)))
    return fam


def gates_of(instr, n: int) -> gl.GateList:
    return gl.from_circuit(build_circuit(instr, n))


def values_for(instr, seed: int) -> list:
    from oracle import qiskit_semantics as oq

    return list(np.random.default_rng(seed).uniform(-math.pi, math.pi, len(oq.parameter_names(instr))))
