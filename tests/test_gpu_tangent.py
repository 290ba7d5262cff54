"""Plain ops of the sweep kernel in tangent form on the GPU (both dtypes): at theta = 0, pi, pi +- 1e-9, 2 pi, random and as
X = u(pi, 0, pi), and a sweep of 32 ops at theta = pi - 1e-12 whose growth the per-sweep budget has to stop (the rest run the
real-top-left body).  Each state against the plan emulator (the same encoded program in NumPy) and the oracle, and through every
consumer of a simulated state: fused diagonal <H>, several observables, exact CVaR, the sampler on the oracle's uniforms and
``Engine.statevector`` of the phase-deferred plan.  tests/test_tangent_plans.py checks on the CPU that the plans hold these ops."""
import numpy as np
import pytest

from oracle import qiskit_semantics as oq
from queasars_b200.operators import SparsePauliOp
from tests import dispatch_coverage as dc
from tests.plan_emulator import run_program
from tests.test_gpu_cvar_exact import assert_cvar
from tests.test_gpu_parity import random_ising, rel_err, tfim
from tests.test_tangent_plans import angle_circuit, budget_circuit

pytestmark = pytest.mark.gpu

CASES = {"angles": (13, lambda: angle_circuit(13, 1)), "budget": (12, lambda: budget_circuit(12, 2))}


@pytest.mark.parametrize("label", sorted(CASES))
@pytest.mark.parametrize("dtype", ["complex128", "complex64"])
def test_plain_ops_in_tangent_form(dtype, label):
    from queasars_b200.engine import Engine

    eng = Engine(device=0, dtype=dtype)
    single = dtype == "complex64"
    tol_sv, tol_ev, tol_cvar = (1e-5, 1e-4, 2e-3) if single else (1e-12, 1e-10, 1e-10)
    n, make = CASES[label]
    instr, values = make()
    gates = dc.gates_of(instr, n)
    want = oq.statevector(instr, n, values)
    probs = np.abs(want) ** 2
    K, R = eng.tile_bits, eng.reg_bits

    # Engine.statevector: the deferred plan against the emulator of its own program, its |psi|^2 against the oracle; the plan as
    # written against the oracle's state
    plan_p = eng.compile(gates, drop_final_phases=True)
    sv = eng.statevector(plan_p, values)
    assert np.all(np.isfinite(sv))
    emu = run_program(dc.plan_for(gates, K, R, True)[1], max(n, K), K, values, reg_bits=R)[: 1 << n]
    assert np.max(np.abs(sv - emu)) < tol_sv
    assert np.max(np.abs(np.abs(sv) ** 2 - probs)) < tol_sv
    plan = eng.compile(gates)
    assert np.max(np.abs(eng.statevector(plan, values) - want)) < tol_sv

    # fused diagonal <H> (one circuit and a batch of both plans), several observables from one state
    diag = random_ising(n, 100 + n)
    table = oq.diagonal_table(n, oq.diag_terms_from_labels(diag))
    ham = eng.hamiltonian(SparsePauliOp.from_list(diag))
    want_d = float(np.dot(probs, table))
    assert rel_err(eng.expectation([plan_p], [values], ham)[0], want_d) < tol_ev
    for g in eng.expectation([plan_p, plan], [values, values], ham):
        assert rel_err(g, want_d) < tol_ev
    rng = np.random.default_rng(n)
    obs = [diag, tfim(n), [("".join(rng.choice(list("IXYZ"), size=n)), float(rng.normal())) for _ in range(6)]]
    got = eng.expectation_many([plan], [values], eng.observables([SparsePauliOp.from_list(o) for o in obs]))[0]
    for g, o in zip(got, obs):
        assert rel_err(g, oq.estimator_expectation(want, o)) < tol_ev

    # exact CVaR of the diagonal Hamiltonian
    for alpha in (0.1, 0.5, 1.0):
        assert_cvar(eng.cvar([plan_p], [values], ham, alpha)[0], probs, table, alpha, tol_cvar)

    # the sampler on the oracle's uniforms: equal draws up to a flip at a CDF boundary (to a neighbouring nonzero state)
    shots = 4000
    u = rng.random(shots)
    got = eng.sample([plan_p], [values], shots, u.reshape(1, -1))[0]
    ref = oq.sample_indices(want, shots, uniforms=u)
    if single:  # complex64 probabilities differ at 1e-7 relative: flips to nearby states
        assert np.count_nonzero(np.abs(got - ref) > 64) <= shots // 100
    else:
        bad = np.nonzero(got != ref)[0]
        assert len(bad) <= 1, len(bad)
        nz = np.flatnonzero(np.abs(emu) ** 2 > 0)
        for i in bad:
            pos = np.searchsorted(nz, ref[i])
            assert got[i] in nz[max(0, pos - 1) : pos + 2], (got[i], ref[i])
    eng.close()
