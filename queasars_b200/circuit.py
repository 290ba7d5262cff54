"""Minimal circuit container exposing the subset of the ``qiskit.circuit.QuantumCircuit`` API that the
gate-list front end (``queasars_b200.gate_list``) reads and that the reference's genome code writes.

Why it exists: Qiskit is not installable in this environment (no network), yet the drop-in boundary
``BaseCircuitEvaluator.evaluate_circuits(circuits, parameter_values)``
(/root/reference/queasars/circuit_evaluation/circuit_evaluation.py:62-87) takes circuit objects.  The front
end is written against the *Qiskit attribute names* (``num_qubits``, ``data``, ``operation.name``,
``operation.params``, ``operation.definition``, ``find_bit(q).index``, ``parameters``, ``assign_parameters``)
so a real ``QuantumCircuit`` and this class go through one and the same code path.

Semantics mirrored from upstream Qiskit: ``parameters`` is sorted by parameter *name* (plain string
compare); a flat value sequence binds in that order; ``decompose()`` expands one level of
``definition``; ``measure_all(inplace=False)`` / ``compose(other, inplace=False)`` return copies.
"""
from __future__ import annotations

import numbers
from typing import Iterable, Mapping, Optional, Sequence, Union


class ParameterExpression:
    """Affine expression ``const + sum_i coeff_i * parameter_i`` (all the hot path needs)."""

    __slots__ = ("_terms", "_const")

    def __init__(self, terms: Mapping["Parameter", float], const: float = 0.0):
        self._terms = {p: float(c) for p, c in terms.items() if c != 0.0}
        self._const = float(const)

    @property
    def parameters(self) -> set:
        return set(self._terms)

    def bind(self, values: Mapping["Parameter", float]):
        terms = {}
        const = self._const
        for prm, coeff in self._terms.items():
            if prm in values:
                const += coeff * float(values[prm])
            else:
                terms[prm] = coeff
        if not terms:
            return const
        return ParameterExpression(terms, const)

    assign = bind

    def __float__(self):
        if self._terms:
            raise TypeError("ParameterExpression with unbound parameters cannot be cast to float")
        return self._const

    # --- affine arithmetic -------------------------------------------------------------------
    @staticmethod
    def _lift(other):
        if isinstance(other, ParameterExpression):
            return other
        if isinstance(other, numbers.Real):
            return ParameterExpression({}, float(other))
        return None

    def __add__(self, other):
        o = self._lift(other)
        if o is None:
            return NotImplemented
        terms = dict(self._terms)
        for p, c in o._terms.items():
            terms[p] = terms.get(p, 0.0) + c
        return ParameterExpression(terms, self._const + o._const)

    __radd__ = __add__

    def __neg__(self):
        return ParameterExpression({p: -c for p, c in self._terms.items()}, -self._const)

    def __sub__(self, other):
        o = self._lift(other)
        if o is None:
            return NotImplemented
        return self + (-o)

    def __rsub__(self, other):
        return (-self) + other

    def __mul__(self, other):
        if not isinstance(other, numbers.Real):
            return NotImplemented
        return ParameterExpression({p: c * other for p, c in self._terms.items()}, self._const * other)

    __rmul__ = __mul__

    def __truediv__(self, other):
        if not isinstance(other, numbers.Real):
            return NotImplemented
        return self * (1.0 / other)

    def __repr__(self):
        parts = [f"{c}*{p.name}" for p, c in self._terms.items()]
        if self._const or not parts:
            parts.append(repr(self._const))
        return " + ".join(parts)


class Parameter(ParameterExpression):
    """Named symbolic parameter; identity is the name (upstream also carries a uuid)."""

    __slots__ = ("_name",)

    def __init__(self, name: str):
        self._name = str(name)
        ParameterExpression.__init__(self, {}, 0.0)
        self._terms = {self: 1.0}

    @property
    def name(self) -> str:
        return self._name

    def __eq__(self, other):
        return isinstance(other, Parameter) and other._name == self._name

    def __hash__(self):
        return hash(("Parameter", self._name))

    def __repr__(self):
        return f"Parameter({self._name})"

    def __reduce__(self):
        return (Parameter, (self._name,))


ParamValue = Union[float, ParameterExpression]


class Qubit:
    __slots__ = ("_index",)

    def __init__(self, index: int):
        self._index = index

    def __repr__(self):
        return f"Qubit({self._index})"


class Clbit:
    """A classical bit; the bits of a ``ClassicalRegister`` know their register and position in it."""

    __slots__ = ("_register", "_index")

    def __init__(self, register: "Optional[ClassicalRegister]" = None, index: Optional[int] = None):
        self._register, self._index = register, index

    def __repr__(self):
        return f"Clbit({self._register.name if self._register is not None else None}, {self._index})"


class ClassicalRegister:
    """``qiskit.circuit.ClassicalRegister(size, name)``: ``size`` fresh clbits, indexable and iterable."""

    _count = 0

    def __init__(self, size: int, name: Optional[str] = None):
        size = int(size)
        if size < 0:
            raise ValueError("a register's size must be non-negative")
        if name is None:
            name = f"c{ClassicalRegister._count}"
            ClassicalRegister._count += 1
        self.name, self.size = str(name), size
        self._bits = [Clbit(self, i) for i in range(size)]

    def __len__(self):
        return self.size

    def __getitem__(self, key):
        return self._bits[key]

    def __iter__(self):
        return iter(self._bits)

    def __repr__(self):
        return f"ClassicalRegister({self.size}, '{self.name}')"


class _BitLocation:
    __slots__ = ("index", "registers")

    def __init__(self, index, registers=None):
        self.index = index
        self.registers = registers or []


class Instruction:
    """``name`` / ``num_qubits`` / ``params`` / ``definition`` like qiskit.circuit.Instruction."""

    def __init__(self, name: str, num_qubits: int, params: Sequence[ParamValue] = (), definition: "Optional[QuantumCircuit]" = None):
        self.name = name
        self.num_qubits = num_qubits
        self.params = list(params)
        self.definition = definition

    def copy(self):
        return type(self).__new__(type(self))._init_from(self)

    def _init_from(self, other):
        self.name, self.num_qubits = other.name, other.num_qubits
        self.params = list(other.params)
        self.definition = other.definition
        return self


class Gate(Instruction):
    pass


class CU3Gate(Gate):
    """qiskit.circuit.library.CU3Gate(theta, phi, lam); qargs = (control, target)."""

    def __init__(self, theta, phi, lam):
        super().__init__("cu3", 2, [theta, phi, lam])


class CircuitInstruction:
    __slots__ = ("operation", "qubits", "clbits")

    def __init__(self, operation: Instruction, qubits: Sequence[Qubit], clbits: Sequence = ()):
        self.operation = operation
        self.qubits = tuple(qubits)
        self.clbits = tuple(clbits)


_STANDARD_ARITY = {
    "id": (1, 0), "x": (1, 0), "y": (1, 0), "z": (1, 0), "h": (1, 0), "s": (1, 0), "sdg": (1, 0), "t": (1, 0),
    "tdg": (1, 0), "sx": (1, 0), "sxdg": (1, 0), "rx": (1, 1), "ry": (1, 1), "rz": (1, 1), "p": (1, 1),
    "u1": (1, 1), "u2": (1, 2), "u3": (1, 3), "u": (1, 3), "cx": (2, 0), "cy": (2, 0), "cz": (2, 0),
    "ch": (2, 0), "cp": (2, 1), "cu1": (2, 1), "crx": (2, 1), "cry": (2, 1), "crz": (2, 1), "cu3": (2, 3),
    "cu": (2, 4), "swap": (2, 0), "rzz": (2, 1), "rxx": (2, 1), "rzx": (2, 1), "ecr": (2, 0),
}  # name -> (n_qubits, n_params)


class QuantumCircuit:
    """``QuantumCircuit(num_qubits)``, ``QuantumCircuit(num_qubits, num_clbits)`` (clbits in one register "c") or
    ``QuantumCircuit(num_qubits, *cregs)`` (``ClassicalRegister``s); a circuit without clbits has no classical registers."""

    def __init__(self, num_qubits: int, *cregs, name: Optional[str] = None):
        if len(cregs) == 1 and isinstance(cregs[0], str):  # QuantumCircuit(n, name): the earlier positional form
            name, cregs = cregs[0], ()
        self.num_qubits = int(num_qubits)
        self.name = name or "circuit"
        self.qubits = [Qubit(i) for i in range(self.num_qubits)]
        self.data: list[CircuitInstruction] = []
        self.global_phase = 0.0
        self.cregs: list[ClassicalRegister] = []
        self.clbits: list[Clbit] = []
        self._clbit_index: dict = {}  # Clbit -> index in self.clbits
        self._b200_version = 0  # bumped by every in-place change that keeps len(data) (plan-cache fingerprint, primitives.py)
        if len(cregs) == 1 and isinstance(cregs[0], numbers.Integral):
            if int(cregs[0]) > 0:
                self.add_register(ClassicalRegister(int(cregs[0]), "c"))
        else:
            for reg in cregs:
                self.add_register(reg)

    # ------------------------------------------------------------------ inspection
    @property
    def num_clbits(self) -> int:
        return len(self.clbits)

    def find_bit(self, bit) -> _BitLocation:
        """Index of a qubit, or index and (register, position) pairs of a clbit, like ``QuantumCircuit.find_bit``."""
        if isinstance(bit, Clbit):
            try:
                index = self._clbit_index[bit]
            except KeyError:
                raise ValueError(f"{bit!r} is not in the circuit") from None
            return _BitLocation(index, [(bit._register, bit._index)] if bit._register is not None else [])
        return _BitLocation(bit._index)

    def add_register(self, register: ClassicalRegister) -> None:
        if not isinstance(register, ClassicalRegister):
            raise TypeError(f"expected a ClassicalRegister, got {type(register).__name__}")
        if any(reg.name == register.name for reg in self.cregs):
            raise ValueError(f'register name "{register.name}" already exists')
        self.cregs.append(register)
        for bit in register:
            if bit not in self._clbit_index:
                self._clbit_index[bit] = len(self.clbits)
                self.clbits.append(bit)

    @property
    def parameters(self) -> list:
        found = set()
        for inst in self.data:
            for prm in inst.operation.params:
                if isinstance(prm, ParameterExpression):
                    found |= prm.parameters
        return sorted(found, key=lambda p: p.name)

    @property
    def num_parameters(self) -> int:
        return len(self.parameters)

    def count_ops(self) -> dict:
        out: dict = {}
        for inst in self.data:
            out[inst.operation.name] = out.get(inst.operation.name, 0) + 1
        return out

    def depth(self) -> int:
        level = [0] * max(1, self.num_qubits)
        for inst in self.data:
            if inst.operation.name == "barrier":
                continue
            idx = [q._index for q in inst.qubits]
            if not idx:
                continue
            d = max(level[i] for i in idx) + 1
            for i in idx:
                level[i] = d
        return max(level)

    def __len__(self):
        return len(self.data)

    # ------------------------------------------------------------------ building
    def _qubit(self, q) -> Qubit:
        if isinstance(q, Qubit):
            return self.qubits[q._index]
        return self.qubits[int(q)]

    def append(self, instruction: Instruction, qargs: Iterable = (), cargs: Iterable = ()):
        qubits = [self._qubit(q) for q in qargs]
        if len(qubits) != instruction.num_qubits:
            raise ValueError(
                f"instruction '{instruction.name}' acts on {instruction.num_qubits} qubits, got {len(qubits)} qargs"
            )
        if len({q._index for q in qubits}) != len(qubits):
            raise ValueError("duplicate qubit arguments")
        self.data.append(CircuitInstruction(instruction, qubits, tuple(self._clbit(c) for c in cargs)))
        return self

    def _clbit(self, c) -> Clbit:
        if isinstance(c, Clbit):
            if c not in self._clbit_index:
                raise ValueError(f"{c!r} is not in the circuit")
            return c
        return self.clbits[int(c)]

    def _bit_list(self, arg, resolve) -> list:
        """One bit or a sequence of them (register, range, list), as ``measure`` accepts them."""
        if isinstance(arg, (ClassicalRegister, range, list, tuple)):
            return [resolve(a) for a in arg]
        return [resolve(arg)]

    def measure(self, qubit, cbit):
        """Measure ``qubit`` into ``cbit``; each may be one bit or a sequence (a register, a range, a list).  One qubit and several
        clbits measures it into each of them; otherwise the two sequences pair up and must have the same length (Qiskit's
        broadcasting)."""
        qubits = self._bit_list(qubit, self._qubit)
        clbits = self._bit_list(cbit, self._clbit)
        if len(qubits) == 1 and len(clbits) > 1:
            qubits = qubits * len(clbits)
        if len(qubits) != len(clbits):
            raise ValueError(f"the amount of qubit({len(qubits)})/clbit({len(clbits)}) arguments does not match the gate expectation")
        for q, c in zip(qubits, clbits):
            self.data.append(CircuitInstruction(Instruction("measure", 1), [q], (c,)))
        return self

    def _std(self, name, qubits, params=()):
        nq, npar = _STANDARD_ARITY[name]
        assert len(qubits) == nq and len(params) == npar
        return self.append(Gate(name, nq, list(params)), qubits)

    def id(self, qubit):
        return self._std("id", [qubit])

    def x(self, qubit):
        return self._std("x", [qubit])

    def y(self, qubit):
        return self._std("y", [qubit])

    def z(self, qubit):
        return self._std("z", [qubit])

    def h(self, qubit):
        return self._std("h", [qubit])

    def s(self, qubit):
        return self._std("s", [qubit])

    def sdg(self, qubit):
        return self._std("sdg", [qubit])

    def t(self, qubit):
        return self._std("t", [qubit])

    def tdg(self, qubit):
        return self._std("tdg", [qubit])

    def sx(self, qubit):
        return self._std("sx", [qubit])

    def rx(self, theta, qubit):
        return self._std("rx", [qubit], [theta])

    def ry(self, theta, qubit):
        return self._std("ry", [qubit], [theta])

    def rz(self, phi, qubit):
        return self._std("rz", [qubit], [phi])

    def p(self, theta, qubit):
        return self._std("p", [qubit], [theta])

    def u(self, theta, phi, lam, qubit):
        return self._std("u", [qubit], [theta, phi, lam])

    def cx(self, control_qubit, target_qubit):
        return self._std("cx", [control_qubit, target_qubit])

    def cz(self, control_qubit, target_qubit):
        return self._std("cz", [control_qubit, target_qubit])

    def cp(self, theta, control_qubit, target_qubit):
        return self._std("cp", [control_qubit, target_qubit], [theta])

    def crz(self, theta, control_qubit, target_qubit):
        return self._std("crz", [control_qubit, target_qubit], [theta])

    def cu(self, theta, phi, lam, gamma, control_qubit, target_qubit):
        return self._std("cu", [control_qubit, target_qubit], [theta, phi, lam, gamma])

    def swap(self, qubit1, qubit2):
        return self._std("swap", [qubit1, qubit2])

    def rzz(self, theta, qubit1, qubit2):
        return self._std("rzz", [qubit1, qubit2], [theta])

    def rxx(self, theta, qubit1, qubit2):
        return self._std("rxx", [qubit1, qubit2], [theta])

    def rzx(self, theta, qubit1, qubit2):
        return self._std("rzx", [qubit1, qubit2], [theta])

    def ecr(self, qubit1, qubit2):
        return self._std("ecr", [qubit1, qubit2])

    def barrier(self, *qargs):
        qubits = [self._qubit(q) for q in qargs] if qargs else list(self.qubits)
        self.data.append(CircuitInstruction(Instruction("barrier", len(qubits)), qubits))
        return self

    # ------------------------------------------------------------------ transformations
    def _empty_like(self, name: Optional[str] = None) -> "QuantumCircuit":
        """Same width, name, phase and classical registers (the same register and clbit objects, as Qiskit's ``copy``); no data."""
        out = QuantumCircuit(self.num_qubits, name=name or self.name)
        out.global_phase = self.global_phase
        for reg in self.cregs:
            out.add_register(reg)
        return out

    def copy(self, name: Optional[str] = None) -> "QuantumCircuit":
        out = self._empty_like(name)
        for inst in self.data:
            op = inst.operation
            new_op = type(op).__new__(type(op))
            Instruction._init_from(new_op, op)
            out.data.append(CircuitInstruction(new_op, [out.qubits[q._index] for q in inst.qubits], inst.clbits))
        return out

    def measure_all(self, inplace: bool = True, add_bits: bool = True):
        """Barrier, then every qubit i measured into clbit i of a new register "meas" (``add_bits``) or of the circuit's own clbits."""
        circ = self if inplace else self.copy()
        if add_bits:
            name = "meas"
            if any(r.name == name for r in circ.cregs):  # (upstream: a fresh name with the same prefix)
                name = f"meas{ClassicalRegister._count}"
                ClassicalRegister._count += 1
            reg = ClassicalRegister(circ.num_qubits, name)
            circ.add_register(reg)
            clbits = list(reg)
        else:
            if circ.num_clbits < circ.num_qubits:
                raise ValueError("The number of classical bits must be equal or greater than the number of qubits.")
            clbits = circ.clbits[: circ.num_qubits]
        circ.barrier()
        circ.measure(list(range(circ.num_qubits)), clbits)
        return None if inplace else circ

    def compose(self, other: "QuantumCircuit", qubits: Optional[Sequence[int]] = None, clbits: Optional[Sequence[int]] = None,
                inplace: bool = False):
        """``other``'s instructions appended on ``qubits`` (default: the first ones) and its clbits mapped onto ``clbits`` (default: the
        first ones) of this circuit, whose registers are kept."""
        if other.num_qubits > self.num_qubits:
            raise ValueError("Trying to compose with another QuantumCircuit which has more 'in' edges.")
        if other.num_clbits > self.num_clbits:
            raise ValueError("Trying to compose with another QuantumCircuit which has more 'out' edges.")
        dest = self if inplace else self.copy()
        mapping = list(range(other.num_qubits)) if qubits is None else [int(q) for q in qubits]
        cmap = list(range(other.num_clbits)) if clbits is None else [dest.find_bit(dest._clbit(c)).index for c in clbits]
        for inst in other.copy().data:
            dest.data.append(
                CircuitInstruction(inst.operation, [dest.qubits[mapping[q._index]] for q in inst.qubits],
                                   tuple(dest.clbits[cmap[other.find_bit(c).index]] for c in inst.clbits))
            )
        dest.global_phase += other.global_phase
        return None if inplace else dest

    def decompose(self) -> "QuantumCircuit":
        out = self._empty_like()
        for inst in self.copy().data:
            definition = inst.operation.definition
            if definition is None:
                out.data.append(CircuitInstruction(inst.operation, [out.qubits[q._index] for q in inst.qubits], inst.clbits))
                continue
            # the operation's params are positionally the definition's (sorted) parameters
            sub = definition
            def_params = sub.parameters
            if def_params and len(inst.operation.params) == len(def_params):
                binding = {p: v for p, v in zip(def_params, inst.operation.params) if not (isinstance(v, Parameter) and v == p)}
                if binding:
                    sub = sub._substitute(binding)
            outer = [q._index for q in inst.qubits]
            for sub_inst in sub.copy().data:
                out.data.append(
                    CircuitInstruction(sub_inst.operation, [out.qubits[outer[q._index]] for q in sub_inst.qubits], sub_inst.clbits)
                )
            out.global_phase += sub.global_phase
        return out

    def _substitute(self, binding: Mapping[Parameter, ParamValue]) -> "QuantumCircuit":
        out = self.copy()
        for inst in out.data:
            op = inst.operation
            new_params = []
            for prm in op.params:
                if isinstance(prm, ParameterExpression) and prm.parameters:
                    expr = ParameterExpression({}, prm._const)
                    for p, c in prm._terms.items():
                        expr = expr + (binding[p] * c if p in binding else ParameterExpression({p: c}))
                    new_params.append(expr if expr.parameters else expr._const)
                else:
                    new_params.append(prm)
            op.params = new_params
            if op.definition is not None and op.definition.parameters:
                op.definition = op.definition._substitute(binding)
        return out

    def assign_parameters(self, parameters, inplace: bool = False, **_ignored):
        params = self.parameters
        if isinstance(parameters, Mapping):
            binding = {}
            for key, val in parameters.items():
                binding[Parameter(key) if isinstance(key, str) else key] = val
        else:
            values = list(parameters)
            if len(values) != len(params):
                raise ValueError(
                    f"Mismatching number of values and parameters. For partial binding please pass a dictionary "
                    f"({len(values)} values for {len(params)} parameters)."
                )
            binding = dict(zip(params, values))
        bound = self._substitute(binding)
        if inplace:
            self.data = bound.data
            self._b200_version += 1
            return None
        return bound


def circuit_to_gate(circuit: QuantumCircuit, label: Optional[str] = None) -> Gate:
    """qiskit.converters.circuit_to_gate: opaque gate whose definition is (a copy of) the circuit."""
    gate = Gate(circuit.name, circuit.num_qubits, list(circuit.parameters), definition=circuit.copy())
    return gate
