"""Reach of the sweep kernel's dispatch table on the CPU: the circuit family of tests/dispatch_coverage.py must hit every body
class, register bit, register pair and branch of ``apply_op`` under every planner configuration the kernels are built for, so
that the GPU tests running it (tests/test_gpu_dispatch.py) cannot silently stop exercising a body when the planner changes.
The plan emulator then reproduces the oracle on these circuits, which makes it the per-plan reference of the GPU tests."""
import numpy as np
import pytest

from oracle import qiskit_semantics as oq
from tests import dispatch_coverage as dc
from tests.plan_emulator import run_program

CONFIGS = [(11, 4), (12, 4), (11, 3)]


@pytest.mark.parametrize("drop", [False, True])
@pytest.mark.parametrize("tile_bits,reg_bits", CONFIGS)
def test_circuit_family_reaches_every_dispatch_class(tile_bits, reg_bits, drop):
    cov = dc.Coverage(reg_bits)
    for n in (13, 14, 15):
        for _, instr in dc.circuit_family(n, tile_bits):
            cov.add(dc.plan_for(dc.gates_of(instr, n), tile_bits, reg_bits, drop)[1])
        cov.add(dc.plan_for(dc.gates_of(dc.zero_start_circuit(n, 5), n), tile_bits, reg_bits, drop, from_zero_state=False)[1])
    print(f"\n(K, R) = ({tile_bits}, {reg_bits}), drop_final_phases={drop}\n{cov.report()}")
    assert cov.missing(drop) == []
    assert all(cov.starts[s] for s in ("zero", "partial", "full"))
    if drop:
        assert not cov.classes[("dense", "real00", "none")]  # phase deferral leaves no uncontrolled gate with phi != 0


@pytest.mark.parametrize("reg_bits", [3, 4])
def test_dispatch_variants_are_distinct_and_decode_to_their_body(reg_bits):
    """The variant numbering (v_dense / v_ctrl / v_diag_* and bits 4, 5) has no collision for either register width, and the
    kernel's branch order in apply_op sends every variant to the body of its class."""
    R = reg_bits
    seen = {}
    for form in ("plain", "real00", "phase"):
        for B in range(R):
            for CB in [None] + [c for c in range(R) if c != B]:
                if form == "plain" and CB is not None:
                    continue
                po = {"kind": 0, "tgt_kind": 1, "tgt_pos": B, "ctrl_kind": 0 if CB is None else 1, "ctrl_pos": 0 if CB is None else CB}
                # (gamma, theta, phi, lam): gamma != 0 -> global phase; gamma == phi == 0 -> real first column
                ang = {"slot": [-1] * 4, "slot2": [-1] * 4, "const": [0.5 if form == "phase" else 0.0, 1.0, 0.0 if form == "plain" else 0.25, 1.0]}
                v = dc.dispatch_variant(po, ang, R)
                assert dc.decode_variant(v, R) == ("dense", form, B, CB)
                seen.setdefault(v, []).append(("dense", form, B, CB))
    for tk in (1, 2, 3):
        for ck in (0, 1, 2, 3):
            po = {"kind": 1, "tgt_kind": tk, "tgt_pos": 1, "ctrl_kind": ck, "ctrl_pos": 2}
            v = dc.dispatch_variant(po, {"slot": [-1] * 4, "slot2": [-1] * 4, "const": [0.1, 0, 0, 0.2]}, R)
            want = ("diag", "gen" if ck == 1 else ("reg" if tk == 1 else "out"), 1 if (tk == 1 and ck != 1) else None, None)
            assert dc.decode_variant(v, R) == want
            seen.setdefault(v, []).append(want)
    for v, bodies in seen.items():
        assert 0 <= v < 64 and len(set(bodies)) == 1, (v, bodies)


@pytest.mark.parametrize("tile_bits,reg_bits", CONFIGS)
def test_emulator_reproduces_the_oracle_on_the_family(tile_bits, reg_bits):
    """Amplitudes to 1e-13 for plans that keep the circuit as written, |psi|^2 to 1e-13 for plans with dropped final phases."""
    checked = 0
    for n in (13, 15):
        fam = dc.circuit_family(n, tile_bits, n_random=1)
        fam.append(("zero", dc.zero_start_circuit(n, 9)))
        for label, instr in fam:
            values = dc.values_for(instr, n)
            want = oq.statevector(instr, n, values)
            gates = dc.gates_of(instr, n)
            zero = label == "zero"
            for drop in (False, True) if not zero else (False,):
                g, enc = dc.plan_for(gates, tile_bits, reg_bits, drop, from_zero_state=not zero)
                got = run_program(enc, max(n, tile_bits), tile_bits, values, reg_bits=reg_bits)
                assert np.max(np.abs(got[1 << n :]), initial=0.0) == 0.0
                got = got[: 1 << n]
                if drop:
                    assert np.max(np.abs(np.abs(got) ** 2 - np.abs(want) ** 2)) < 1e-13, label
                else:
                    assert np.max(np.abs(got - want)) < 1e-13, label
                checked += 1
    assert checked >= 10
