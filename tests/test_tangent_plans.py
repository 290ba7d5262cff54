"""Circuits for the tangent form of the sweep kernel's plain ops (uncontrolled dense gates with a real first column, run as
c * [[1, -t E], [t, E]] with t = tan(theta / 2) and the c's restored by one scale per sweep), and CPU checks that their plans
put those ops where the GPU tests (tests/test_gpu_tangent.py) need them.  The kernel keeps an op in tangent form only while the
product of the |c|'s of the sweep's plain ops stays >= 2^-400 (complex128) / 2^-40 (complex64); the others run the
real-top-left body with their matrix as bound."""
import math

import numpy as np

from queasars_b200 import engine as qe
from queasars_b200 import gate_list as gl
from tests import dispatch_coverage as dc

# theta of the plain ops: identity, pi (c = 6e-17, not 0), either side of pi, 2 pi (c = -1: a negative scale)
SPECIAL_THETAS = (0.0, math.pi, math.pi + 1e-9, math.pi - 1e-9, 2 * math.pi)
NEAR_PI = math.pi - 1e-12  # t ~ 2^41: nine of them exhaust the complex128 budget, one the complex64 one


class _Names:
    """Parameter names in slot order (name-sorted) with their values."""

    def __init__(self):
        self.values = []

    def __call__(self, v):
        self.values.append(float(v))
        return f"p{len(self.values) - 1:03d}"


def angle_circuit(n: int, seed: int):
    """Plain ops at the special angles, at random angles and X = u(pi, 0, pi) on every qubit, between layers of cu3."""
    rng = np.random.default_rng(seed)
    par = _Names()
    instr = [("ry", (q,), (float(rng.uniform(0.2, 3.0)),)) for q in range(n)]  # product start
    for rep in range(3):
        for q in range(n):
            k = (q + rep) % 8
            if k == 7:
                instr.append(("u", (q,), (math.pi, 0.0, math.pi)))
                continue
            theta = SPECIAL_THETAS[k] if k < len(SPECIAL_THETAS) else rng.uniform(-math.pi, math.pi)
            instr.append(("u", (q,), (par(theta), par(rng.uniform(-math.pi, math.pi)), par(rng.uniform(-math.pi, math.pi)))))
        for q in range(n):
            instr.append(("cu3", (q, (q + 1 + rep) % n), tuple(par(rng.uniform(-math.pi, math.pi)) for _ in range(3))))
    return instr, par.values


def budget_circuit(n: int, seed: int, count: int = 32):
    """``count`` plain ops at theta = pi - 1e-12 on four qubits, behind an entangling layer: in tangent form all of them would
    grow the amplitudes by 2^(41 count), far past the double range; then cu3 and random plain ops."""
    rng = np.random.default_rng(seed)
    par = _Names()
    instr = [("ry", (q,), (float(rng.uniform(0.2, 3.0)),)) for q in range(n)]
    instr += [("cu3", (q, (q + 1) % 4), tuple(par(rng.uniform(-math.pi, math.pi)) for _ in range(3))) for q in range(4)]
    for i in range(count):
        instr.append(("u", (i % 4,), (par(NEAR_PI), par(rng.uniform(-math.pi, math.pi)), par(rng.uniform(-math.pi, math.pi)))))
    instr += [("cu3", (q, q + 1), tuple(par(rng.uniform(-math.pi, math.pi)) for _ in range(3))) for q in range(n - 1)]
    instr += [("u", (q,), tuple(par(rng.uniform(-math.pi, math.pi)) for _ in range(3))) for q in range(n)]
    return instr, par.values


def plain_ops_per_sweep(instr, n: int, tile_bits: int = 11, reg_bits: int = 4, drop: bool = True) -> list:
    """Number of plain-class pass ops in each sweep of the plan the engine compiles for ``instr``."""
    _, enc = dc.plan_for(dc.gates_of(instr, n), tile_bits, reg_bits, drop)
    sweeps, passes, pass_ops, angles, _ = enc
    out = []
    for sw in sweeps:
        lo, hi = int(passes[int(sw["pass_begin"])]["op_begin"]), int(passes[int(sw["pass_end"]) - 1]["op_end"])
        out.append(sum(dc.classify(po, angles[int(po["op_index"])])["cls"] == ("dense", "plain", "none") for po in pass_ops[lo:hi]))
    return out


def test_angle_circuit_runs_plain_ops():
    # with its final phases deferred (dropped) every u of the circuit is a plain op, spread over more than one sweep
    counts = plain_ops_per_sweep(angle_circuit(13, 1)[0], 13)
    assert sum(counts) == 3 * 13 and sum(c > 0 for c in counts) >= 2, counts


def test_budget_circuit_holds_twenty_near_pi_ops_in_one_sweep():
    instr, values = budget_circuit(12, 2)
    assert max(plain_ops_per_sweep(instr, 12)) >= 20
    # what the kernel's budget admits of them: nine in double (2^-41 each against 2^-400), none in single
    c = math.cos(NEAR_PI / 2)
    assert math.floor(400 / -math.log2(c)) == 9 and c < 2.0**-40


def test_fp64_count_of_the_plain_class():
    gates = dc.gates_of([("u", (0,), ("a", "b", "c")), ("cu3", (0, 1), ("a", "b", "c"))], 2)
    ops = qe.rewritten(gates, True).ops
    plain = [op for op in ops if op.kind == gl.DENSE and op.control < 0 and op.phi.is_zero and op.gamma.slot < 0 and op.gamma.const == 0.0]
    assert plain and all(gl.dfma_per_amplitude(op) == 4.0 for op in plain)
    assert all(gl.dfma_per_amplitude(op) == 3.5 for op in ops if op.kind == gl.DENSE and op.control >= 0 and op.gamma.slot < 0 and op.gamma.const == 0.0)
