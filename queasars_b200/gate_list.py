"""Transpile-to-gate-list front end: circuit object -> flat list of kernel-level operations.

This replaces, for the B200 path, the per-call ``PassManager.run`` + ``EstimatorPub.coerce`` + parameter
binding the reference performs on every objective call
(/root/reference/queasars/circuit_evaluation/transpiling_primitives.py:47, 73-80;
circuit_evaluation.py:204-213).  A circuit is parsed ONCE into a ``GateList`` whose angles are affine
functions of parameter *slots*; binding then happens on the device from the flat parameter vector.

Binding order: slot ``i`` is ``circuit.parameters[i]`` -- upstream that view is sorted by parameter name
(plain string compare), which is why a flat ``list[float]`` binds (lambda, phi, theta) per gate and
``q10`` before ``q1_`` (SURVEY.md section 3.4).  The front end never re-sorts: it trusts
``circuit.parameters`` of whatever circuit class it is given (real Qiskit or ``queasars_b200.circuit``).

Kernel-level operation set (everything lowers to these two):
  DENSE  target, optional control: 2x2 matrix  e^{i gamma} * U(theta, phi, lam)
  DIAG   target, optional control: diag(e^{i gamma}, e^{i (gamma + lam)})
with ``U(theta,phi,lam) = [[cos, -e^{i lam} sin], [e^{i phi} sin, e^{i(phi+lam)} cos]]`` (half angle), the
``u`` gate the EVQE genome emits (evqe/quantum_circuit/quantum_gate.py:96-102; ``cu3`` :157-165 is the same
matrix on the control=1 subspace, qargs = (control, target)).
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Optional, Sequence

DENSE = 0
DIAG = 1


class UnsupportedCircuitError(ValueError):
    """Raised for instructions the gate-list front end cannot lower."""


@dataclass(frozen=True)
class Angle:
    """value = const + coeff * params[slot] + coeff2 * params[slot2]   (slot == -1: no such term).  Circuits hand in angles
    with one parameter; the second term appears when the phase-deferral rewrite (``defer_phases``) adds the trailing phase of
    the previous gate on a qubit to the next gate's angles."""

    slot: int = -1
    coeff: float = 0.0
    const: float = 0.0
    slot2: int = -1
    coeff2: float = 0.0

    def scaled(self, s: float) -> "Angle":
        return Angle(self.slot, self.coeff * s, self.const * s, self.slot2, self.coeff2 * s)

    def shifted(self, c: float) -> "Angle":
        return Angle(self.slot, self.coeff, self.const + c, self.slot2, self.coeff2)

    def value(self, params: Sequence[float]) -> float:
        v = self.const + (self.coeff * params[self.slot] if self.slot >= 0 else 0.0)
        return v + (self.coeff2 * params[self.slot2] if self.slot2 >= 0 else 0.0)

    @property
    def is_zero(self) -> bool:
        return self.slot < 0 and self.slot2 < 0 and self.const == 0.0

    def plus(self, other: "Angle", sign: float = 1.0) -> Optional["Angle"]:
        """self + sign * other, or None when the sum would need more than two parameter terms."""
        terms: dict = {}
        for sl, cf in ((self.slot, self.coeff), (self.slot2, self.coeff2), (other.slot, sign * other.coeff), (other.slot2, sign * other.coeff2)):
            if sl >= 0 and cf != 0.0:
                terms[sl] = terms.get(sl, 0.0) + cf
        terms = [(sl, cf) for sl, cf in terms.items() if cf != 0.0]
        if len(terms) > 2:
            return None
        terms += [(-1, 0.0)] * (2 - len(terms))
        return Angle(terms[0][0], terms[0][1], self.const + sign * other.const, terms[1][0], terms[1][1])


ZERO = Angle()


def const(v: float) -> Angle:
    return Angle(-1, 0.0, float(v))


@dataclass(frozen=True)
class KernelOp:
    kind: int  # DENSE | DIAG
    target: int
    control: int  # -1: none
    gamma: Angle = ZERO
    theta: Angle = ZERO
    phi: Angle = ZERO
    lam: Angle = ZERO

    @property
    def angles(self) -> tuple[Angle, Angle, Angle, Angle]:
        return (self.gamma, self.theta, self.phi, self.lam)

    @property
    def qubits(self) -> tuple[int, ...]:
        return (self.target,) if self.control < 0 else (self.target, self.control)

    def matrix(self, params: Sequence[float]):
        """2x2 matrix as nested tuples (host-side helper for tests / plan emulation)."""
        import cmath

        g, t, p, l = (a.value(params) for a in self.angles)
        if self.kind == DIAG:
            return ((cmath.exp(1j * g), 0j), (0j, cmath.exp(1j * (g + l))))
        c, s = math.cos(t / 2), math.sin(t / 2)
        return (
            (cmath.exp(1j * g) * c, -cmath.exp(1j * (g + l)) * s),
            (cmath.exp(1j * (g + p)) * s, cmath.exp(1j * (g + p + l)) * c),
        )


def defer_phases(ops: Sequence[KernelOp], drop_final: bool = False) -> list[KernelOp]:
    """Exact rewrite  e^{i gamma} U(theta, phi, lam) = e^{i gamma} D(phi) R_Y(theta) D(lam),  D(a) = diag(1, e^{ia}):  the trailing
    D(phi) of every UNCONTROLLED dense gate is not applied but kept as a pending phase P_q on its qubit.  Diagonals commute
    with controls and with each other, so the pending phase travels forward until
      * the next uncontrolled dense gate on q absorbs it:     U(theta, phi, lam) D(P) = D(phi) [R_Y(theta) D(lam + P)]
      * a controlled dense gate TARGETING q lets it through:  CU(theta, phi, lam) D_q(P) = D_q(P) CU(theta, phi - P, lam + P)
      * the circuit ends: one DIAG op per qubit with a non-zero pending phase -- or nothing when ``drop_final`` (the caller
        only needs |psi_k|^2: diagonal observables and sampling cannot see a diagonal phase).
    Every emitted uncontrolled dense gate then has phi == 0: its matrix [[c, -s e^{i lam}], [s, c e^{i lam}]] has a real first
    column and costs 12 instead of 14 multiply-adds per amplitude pair in the sweep kernel (REAL10 variants); `u -> u` chains
    on a qubit never pay for the intermediate phase at all.  Angles stay affine in at most two parameters (the pending phase is
    always the ORIGINAL phi of one gate); where a sum would need three, the pending phase is materialised as a DIAG op first."""
    pending: dict[int, Angle] = {}
    out: list[KernelOp] = []

    def flush(q: int) -> None:
        p = pending.pop(q, None)
        if p is not None and not p.is_zero:
            out.append(_diag(q, lam=p))

    for op in ops:
        if op.kind != DENSE:
            out.append(op)  # diagonal on everything it touches: commutes with every pending phase
            continue
        t = op.target
        p = pending.get(t, ZERO)
        if op.control < 0:
            lam = op.lam.plus(p)
            if lam is None:
                flush(t)
                lam = op.lam
            out.append(KernelOp(DENSE, t, -1, op.gamma, op.theta, ZERO, lam))
            pending[t] = op.phi
        else:
            phi, lam = op.phi.plus(p, -1.0), op.lam.plus(p)
            if phi is None or lam is None:
                flush(t)
                phi, lam = op.phi, op.lam
            out.append(KernelOp(DENSE, t, op.control, op.gamma, op.theta, phi, lam))
    if not drop_final:
        for q in sorted(pending):
            flush(q)
    return out


def dfma_per_amplitude(op: KernelOp) -> float:
    """FP64 multiply-add-class instructions per amplitude the sweep kernel spends on ``op`` (roofline accounting in bench.py,
    sweep balancing in the planner): a dense 2x2 gate costs 16 per amplitude pair, 14 when its top-left entry is real (no global
    phase); an uncontrolled one whose bottom-left entry is real as well (phi == 0: the R_Y * D form of the phase-deferred front
    end) runs in tangent form, c * [[1, -t E], [t, E]], at 8 per pair, its c folded into one scale per sweep (2 per amplitude,
    not counted here; the rare op over the sweep's growth budget runs the 14 body instead); a diagonal 4 per amplitude it
    touches; a controlled op touches half of the amplitudes."""
    if op.kind == DIAG:
        per = 4.0
    else:
        real00 = op.gamma.slot < 0 and op.gamma.const == 0.0
        plain = real00 and op.phi.is_zero and op.control < 0  # only uncontrolled gates have the tangent body
        per = 4.0 if plain else (7.0 if real00 else 8.0)
    return per * (1.0 if op.control < 0 else 0.5)


@dataclass
class GateList:
    n_qubits: int
    ops: list[KernelOp] = field(default_factory=list)
    n_params: int = 0
    param_names: tuple[str, ...] = ()

    def structure_key(self) -> tuple:
        return (self.n_qubits, self.n_params, tuple(self.ops))


HALF_PI = math.pi / 2


def _dense(t, c=-1, gamma=ZERO, theta=ZERO, phi=ZERO, lam=ZERO):
    return KernelOp(DENSE, t, c, gamma, theta, phi, lam)


def _diag(t, c=-1, gamma=ZERO, lam=ZERO):
    return KernelOp(DIAG, t, c, gamma, ZERO, ZERO, lam)


def _h(t, c=-1):
    return _dense(t, c, theta=const(HALF_PI), lam=const(math.pi))


def _x(t, c=-1):
    return _dense(t, c, theta=const(math.pi), lam=const(math.pi))


def _rzz(a: Angle, q0: int, q1: int) -> list[KernelOp]:
    # parity phase: rz(a) on q0, then on the q1=1 subspace diag(e^{ia}, e^{-ia}) on q0
    return [_diag(q0, gamma=a.scaled(-0.5), lam=a), _diag(q0, q1, gamma=a, lam=a.scaled(-2.0))]


def lower_instruction(name: str, q: Sequence[int], a: Sequence[Angle]) -> list[KernelOp]:
    """Lower one named gate to kernel ops (exact including global phase; ``q`` = qargs in Qiskit order)."""
    if name in ("id", "i", "barrier", "measure", "delay"):
        return []
    if name in ("u", "u3"):
        return [_dense(q[0], theta=a[0], phi=a[1], lam=a[2])]
    if name == "u2":
        return [_dense(q[0], theta=const(HALF_PI), phi=a[0], lam=a[1])]
    if name in ("p", "u1"):
        return [_diag(q[0], lam=a[0])]
    if name == "rz":
        return [_diag(q[0], gamma=a[0].scaled(-0.5), lam=a[0])]
    if name == "rx":
        return [_dense(q[0], theta=a[0], phi=const(-HALF_PI), lam=const(HALF_PI))]
    if name == "ry":
        return [_dense(q[0], theta=a[0])]
    if name == "x":
        return [_x(q[0])]
    if name == "y":
        return [_dense(q[0], theta=const(math.pi), phi=const(HALF_PI), lam=const(HALF_PI))]
    if name == "z":
        return [_diag(q[0], lam=const(math.pi))]
    if name == "h":
        return [_h(q[0])]
    if name == "s":
        return [_diag(q[0], lam=const(HALF_PI))]
    if name == "sdg":
        return [_diag(q[0], lam=const(-HALF_PI))]
    if name == "t":
        return [_diag(q[0], lam=const(math.pi / 4))]
    if name == "tdg":
        return [_diag(q[0], lam=const(-math.pi / 4))]
    if name == "sx":
        return [_dense(q[0], gamma=const(math.pi / 4), theta=const(HALF_PI), phi=const(-HALF_PI), lam=const(HALF_PI))]
    if name == "sxdg":
        return [_dense(q[0], gamma=const(-math.pi / 4), theta=const(-HALF_PI), phi=const(-HALF_PI), lam=const(HALF_PI))]
    # controlled gates: qargs = (control, target)
    if name == "cx":
        return [_x(q[1], q[0])]
    if name == "cy":
        return [_dense(q[1], q[0], theta=const(math.pi), phi=const(HALF_PI), lam=const(HALF_PI))]
    if name == "cz":
        return [_diag(q[1], q[0], lam=const(math.pi))]
    if name == "ch":
        return [_h(q[1], q[0])]
    if name in ("cp", "cu1"):
        return [_diag(q[1], q[0], lam=a[0])]
    if name == "crz":
        return [_diag(q[1], q[0], gamma=a[0].scaled(-0.5), lam=a[0])]
    if name == "crx":
        return [_dense(q[1], q[0], theta=a[0], phi=const(-HALF_PI), lam=const(HALF_PI))]
    if name == "cry":
        return [_dense(q[1], q[0], theta=a[0])]
    if name == "cu3":
        return [_dense(q[1], q[0], theta=a[0], phi=a[1], lam=a[2])]
    if name == "cu":
        return [_dense(q[1], q[0], gamma=a[3], theta=a[0], phi=a[1], lam=a[2])]
    if name == "swap":
        return [_x(q[1], q[0]), _x(q[0], q[1]), _x(q[1], q[0])]
    if name == "rzz":
        return _rzz(a[0], q[0], q[1])
    if name == "rzx":  # Z on q[0], X on q[1]
        return [_h(q[1])] + _rzz(a[0], q[0], q[1]) + [_h(q[1])]
    if name == "rxx":
        return [_h(q[0]), _h(q[1])] + _rzz(a[0], q[0], q[1]) + [_h(q[0]), _h(q[1])]
    if name == "ecr":
        return (
            lower_instruction("rzx", q, [const(math.pi / 4)])
            + [_x(q[0])]
            + lower_instruction("rzx", q, [const(-math.pi / 4)])
        )
    raise UnsupportedCircuitError(f"gate '{name}' is not supported by the B200 gate-list front end")


class _NeedsHostBinding(Exception):
    pass


def _to_angle(param, slot_of: dict) -> Angle:
    params = getattr(param, "parameters", None)
    if not params:
        return const(float(param))
    params = list(params)
    if len(params) != 1:
        raise _NeedsHostBinding
    prm = params[0]
    if getattr(param, "name", None) is not None and param == prm:  # a bare Parameter
        return Angle(slot_of[prm], 1.0, 0.0)
    try:
        f0 = float(param.bind({prm: 0.0}))
        f1 = float(param.bind({prm: 1.0}))
        f2 = float(param.bind({prm: 2.5}))
    except Exception as exc:  # non-real / unbindable expression
        raise _NeedsHostBinding from exc
    coeff = f1 - f0
    if abs(f0 + 2.5 * coeff - f2) > 1e-12 * max(1.0, abs(f2)):
        raise _NeedsHostBinding  # not affine (e.g. sin(p)): bind on the host instead
    return Angle(slot_of[prm], coeff, f0)


def _walk(circuit, qubit_map: Optional[list[int]], slot_of: dict, out: list[KernelOp]) -> None:
    for inst in circuit.data:
        op = inst.operation
        qubits = [circuit.find_bit(qb).index for qb in inst.qubits]
        if qubit_map is not None:
            qubits = [qubit_map[i] for i in qubits]
        name = op.name
        definition = None
        try:
            out.extend(lower_instruction(name, qubits, [_to_angle(p, slot_of) for p in op.params]))
            continue
        except UnsupportedCircuitError:
            definition = getattr(op, "definition", None)
            if definition is None:
                raise
        if any(getattr(p, "parameters", None) for p in op.params) and list(op.params) != list(definition.parameters):
            raise _NeedsHostBinding  # re-parameterised composite gate: let the circuit class resolve it
        _walk(definition, qubits, slot_of, out)


def from_circuit(circuit) -> GateList:
    """Parse a (Qiskit-API) circuit.  Composite instructions are expanded through ``definition``;
    ``barrier``/``measure``/``id`` emit nothing; the global phase is dropped (it cannot influence
    expectation values or sampled distributions)."""
    parameters = list(circuit.parameters)
    slot_of = {p: i for i, p in enumerate(parameters)}
    ops: list[KernelOp] = []
    _walk(circuit, None, slot_of, ops)
    return GateList(
        n_qubits=int(circuit.num_qubits),
        ops=ops,
        n_params=len(parameters),
        param_names=tuple(getattr(p, "name", str(p)) for p in parameters),
    )


def from_circuit_or_none(circuit) -> Optional[GateList]:
    """``None`` when some angle is not an affine function of a single parameter: the caller then binds on
    the host per call (``circuit.assign_parameters(values)``) and parses the numeric circuit."""
    try:
        return from_circuit(circuit)
    except _NeedsHostBinding:
        return None


# -------------------------------------------------------------------------------------------------
# direct genome -> gate list path (SURVEY.md section 8f-3): bypasses QuantumCircuit construction
# -------------------------------------------------------------------------------------------------
def from_evqe_individual(individual, parameterized_layers: Optional[set] = None) -> GateList:
    """Gate list of ``individual.get_partially_parameterized_quantum_circuit(parameterized_layers)``
    (/root/reference/queasars/minimum_eigensolvers/evqe/evolutionary_algorithm/individual.py:288-322)
    without building a circuit.  Works on the reference's ``EVQEIndividual`` by duck typing
    (``layers[i].gates[q]`` with ``qubit_index`` / ``control_qubit_index``, ``parameter_values``,
    ``layer_parameter_indices``).  Slots follow the name-sorted order the circuit would have."""
    layers = individual.layers
    n_layers = len(layers)
    n_qubits = individual.n_qubits
    if parameterized_layers is None:
        parameterized = set(range(n_layers))
    else:
        parameterized = {i % n_layers for i in parameterized_layers}

    def gate_names(layer_id: int, layer) -> list[tuple[str, object]]:
        found = []
        for gate in layer.gates:
            if type(gate).n_parameters() == 3:
                pre = f"layer{layer_id}_q{gate.qubit_index}_"
                found.append((pre, gate))
        return found

    names: list[str] = []
    for i in sorted(parameterized):
        for pre, _ in gate_names(i, layers[i]):
            names += [pre + "theta", pre + "phi", pre + "lambda"]
    names.sort()
    slot = {nm: k for k, nm in enumerate(names)}

    ops: list[KernelOp] = []
    for i, layer in enumerate(layers):
        rotating = gate_names(i, layer)
        if i in parameterized:
            table = {pre: (Angle(slot[pre + "theta"], 1.0, 0.0), Angle(slot[pre + "phi"], 1.0, 0.0), Angle(slot[pre + "lambda"], 1.0, 0.0)) for pre, _ in rotating}
        else:
            # genome-order stored values bind positionally onto the layer's name-sorted parameters
            # (circuit_layer.py:233-235)
            stored = [individual.parameter_values[j] for j in individual.layer_parameter_indices[i]]
            layer_names = sorted(pre + suffix for pre, _ in rotating for suffix in ("theta", "phi", "lambda"))
            value = dict(zip(layer_names, stored))
            table = {pre: (const(value[pre + "theta"]), const(value[pre + "phi"]), const(value[pre + "lambda"])) for pre, _ in rotating}
        for pre, gate in rotating:
            th, ph, la = table[pre]
            control = getattr(gate, "control_qubit_index", -1)
            ops.append(_dense(gate.qubit_index, control, theta=th, phi=ph, lam=la))
    return GateList(n_qubits=n_qubits, ops=ops, n_params=len(names), param_names=tuple(names))
