"""Exact (shot-free) CVaR of a statevector sharded over several GPUs (``LocalShardedStatevector.cvar``: the sort-free weighted
select of ``cvar_select_kernel``) against the definition on the oracle state and against the single-GPU ``Engine.cvar``, its
determinism, its scratch bound, and the sampler evaluators with ``sampler_shots=None`` at sharded widths.  On a one-GPU box the
shards are virtual (several shards on one device), as in test_gpu_sharded_local.py.  Knife-edge stops are accepted as in
test_gpu_cvar_exact.py."""
import math

import numpy as np
import pytest

from oracle import c_oracle
from oracle import qiskit_semantics as oq
from queasars_b200 import expectation as ex
from queasars_b200 import gate_list as gl
from queasars_b200.operators import SparsePauliOp
from tests.test_gpu_cvar_exact import accepted_values, assert_cvar, evqe_case, jssp_op, probs_of
from tests.test_gpu_parity import random_ising
from tests.test_gpu_sharded_local import shard_engines

pytestmark = pytest.mark.gpu

ALPHAS = (0.05, 0.25, 0.5, 0.9, 1.0)


def diag_of(terms):
    d = oq.diag_terms_from_labels(terms)
    return [z for z, _ in d], [c for _, c in d]


def sharded_run(n, shards, circ, values, engines=None):
    from queasars_b200.sharded import LocalShardedStatevector

    sv = LocalShardedStatevector(n, engines or shard_engines(shards), min_local=8)
    sv.run(gl.from_circuit(circ), values)
    return sv


def stop_of(probs, energies, alpha):
    order = np.arange(probs.size) if ex._close(alpha, 1) else np.argsort(energies, kind="stable")
    cum = np.cumsum(probs[order])
    return int(order[np.nonzero(cum >= alpha - (1e-8 + 1e-5 * alpha))[0][0]])


@pytest.mark.parametrize("n,shards", [(14, 1), (15, 2), (16, 4), (18, 8)])
def test_random_ising_against_the_oracle(n, shards):
    terms = random_ising(n, 11 + n)
    z, c = diag_of(terms)
    energies = oq.diagonal_table(n, list(zip(z, c)))
    for s in range(3):
        instr, values, circ = evqe_case(n, 3 + s, 5100 + 17 * n + s)
        sv = sharded_run(n, shards, circ, values)
        if shards > 1:
            assert sv.position != list(range(n))  # logical bits are read from permuted physical positions
        probs = probs_of(instr, n, values)
        for alpha in ALPHAS:
            value, stop = sv.cvar(z, c, alpha)
            assert_cvar(value, probs, energies, alpha, 1e-10)
            if len(accepted_values(probs, energies, alpha)) == 1:
                assert stop == stop_of(probs, energies, alpha)
        sv.close()


@pytest.mark.parametrize("shards", [1, 2, 4, 8])
def test_jssp_12q_stop_index_inside_ties(jssp_golden, shards):
    """jssp_12q's terms on the low 12 of 16 qubits (a shard must hold at least one 2^11-amplitude sweep tile); the 4 spectator
    qubits multiply every tie run by 16."""
    _, diag_terms = jssp_op(jssp_golden["jssp_12q"])
    n = 16
    z, c = [t[0] for t in diag_terms], [t[1] for t in diag_terms]
    energies = oq.diagonal_table(n, diag_terms)
    ties = 0
    for s in range(4):
        instr, values, circ = evqe_case(n, 3 + s % 3, 900 + s)
        sv = sharded_run(n, shards, circ, values)
        probs = probs_of(instr, n, values)
        for alpha in ALPHAS:
            value, stop = sv.cvar(z, c, alpha)
            assert_cvar(value, probs, energies, alpha, 1e-10)
            if len(accepted_values(probs, energies, alpha)) == 1:
                want = stop_of(probs, energies, alpha)
                assert stop == want
                ties += int(np.count_nonzero(energies == energies[want])) > 1
        sv.close()
    assert ties  # the degenerate JSSP spectrum puts stops inside runs of tied energies


@pytest.mark.parametrize("shards", [2, 4])
def test_against_the_single_gpu_route(shards, jssp_golden):
    from queasars_b200.primitives import get_engine

    engine = get_engine(0)
    cases = [(20, SparsePauliOp.from_list(random_ising(20, 3)), evqe_case(20, 4, 77))]
    op26, _ = jssp_op(jssp_golden["jssp_26q"])
    cases.append((26, op26, evqe_case(26, 4, 26)))
    for n, op, (instr, values, circ) in cases:
        ham = engine.hamiltonian(op, build_table=False)
        plan = engine.compile(gl.from_circuit(circ), drop_final_phases=True)
        sv = sharded_run(n, shards, circ, values)
        state = sv.gather_logical()
        probs = state.real**2 + state.imag**2
        del state
        energies = c_oracle.diag_table(n, list(zip(ham.z_masks.tolist(), ham.coeffs.tolist())))
        for alpha in (0.05, 0.5, 1.0):
            single = engine.cvar([plan], [values], ham, alpha)[0]
            value, _ = sv.cvar(ham.z_masks, ham.coeffs, alpha)
            cands = accepted_values(probs, energies, alpha)
            if len(cands) == 1:
                assert abs(value - single) <= 1e-10 * max(1.0, abs(single)), (n, alpha, value, single)
            assert_cvar(value, probs, energies, alpha, 1e-10)
        sv.close()


def test_bit_identical_across_calls():
    n = 16
    z, c = diag_of(random_ising(n, 9))
    _, values, circ = evqe_case(n, 4, 314)
    sv = sharded_run(n, 4, circ, values)
    for alpha in (0.1, 0.5, 1.0):
        a, b = sv.cvar(z, c, alpha), sv.cvar(z, c, alpha)
        assert np.float64(a[0]).tobytes() == np.float64(b[0]).tobytes() and a[1] == b[1]
    sv.close()


def test_scratch_does_not_grow_with_the_shard():
    """Engines whose workspace limit is a few MiB beyond the two shard buffers: the select needs only O(buckets x CTAs) scratch."""
    import torch

    from queasars_b200 import _native
    from queasars_b200.engine import Engine
    from queasars_b200.sharded import LocalShardedStatevector

    n, shards = 24, 4
    n_dev = min(_native.device_count(), shards)
    shard_bytes = 16 << (n - 2)
    per_device = 2 * shard_bytes * (shards // n_dev)
    engines = [Engine(device=d, workspace_limit=per_device + (4 << 20)) for d in range(n_dev)]
    instr, values, circ = evqe_case(n, 3, 2424)
    sv = LocalShardedStatevector(n, [engines[r % n_dev] for r in range(shards)], min_local=8)
    sv.run(gl.from_circuit(circ), values)
    z, c = diag_of(random_ising(n, 2))
    free_before = torch.cuda.mem_get_info(0)[0]
    value, _ = sv.cvar(z, c, 0.3)
    used = free_before - torch.cuda.mem_get_info(0)[0]
    assert used <= 8 << 20, f"the select allocated {used} bytes on device 0"
    probs = probs_of(instr, n, values)
    assert_cvar(value, probs, c_oracle.diag_table(n, list(zip(z, c))), 0.3, 1e-10)
    assert 1 <= sv.cvar_passes <= 8 + math.ceil(n / 8)
    sv.close()


@pytest.mark.parametrize("alpha", [0.2, 1.0])
def test_sampler_evaluators_at_sharded_widths(alpha):
    from queasars_b200 import B200SamplerV2, DiagonalEnergyBitstringEvaluator
    from queasars_b200.evaluators import B200BitstringCircuitEvaluator, B200OperatorSamplerCircuitEvaluator

    n = 15
    terms = random_ising(n, 6)
    op = SparsePauliOp.from_list(terms)
    z, c = diag_of(terms)
    energies = oq.diagonal_table(n, list(zip(z, c)))
    cases = [evqe_case(n, 3, 60 + s) for s in range(3)]
    circuits, params = [cc for _, _, cc in cases], [v for _, v, _ in cases]
    smp = B200SamplerV2(devices="all", coalesce=False, shard_min_qubits=14)
    smp._engines_obj = shard_engines(4)
    ref = B200SamplerV2(device=0, coalesce=False)
    bits = DiagonalEnergyBitstringEvaluator(n, z, c)
    for kind, make in (("operator", lambda s: B200OperatorSamplerCircuitEvaluator(s, None, op, alpha)),
                       ("bitstring", lambda s: B200BitstringCircuitEvaluator(s, None, bits, alpha))):
        got = make(smp).evaluate_circuits(circuits, params)
        want = make(ref).evaluate_circuits(circuits, params)
        for g, w, (instr, values, _) in zip(got, want, cases):
            probs = probs_of(instr, n, values)
            if kind == "operator" and alpha == 1.0:  # <H> itself (the diagonal expectation of the sharded state)
                exact = float(np.dot(probs, energies))
                assert abs(g - exact) <= 1e-10 * max(1.0, abs(exact)) and abs(g - w) <= 1e-10 * max(1.0, abs(w))
                continue
            if len(accepted_values(probs, energies, alpha)) == 1:
                assert abs(g - w) <= 1e-10 * max(1.0, abs(w))
            assert_cvar(g, probs, energies, alpha, 1e-10)
    assert smp._sharded_obj[n].world == 4


def test_35_qubits_on_8_gpus_closed_form():
    """Product state RY(theta) on every qubit, H = sum_q Z_q: E = n - 2 j on the C(n, j) states with j ones, each of
    probability s^j (1 - s)^(n - j), s = sin^2(theta / 2).  The lower tail fills the levels from j = n down; the greedy fill
    and the closed form filled exactly to the stop bound differ by at most |E| p_max / alpha."""
    from queasars_b200 import QuantumCircuit, _native
    from queasars_b200.primitives import get_engine
    from queasars_b200.sharded import LocalShardedStatevector

    if _native.device_count() < 8:
        pytest.skip("35 qubits need 8 GPUs")
    n, theta = 35, 1.9
    circ = QuantumCircuit(n)
    for q in range(n):
        circ.ry(theta, q)
    sv = LocalShardedStatevector(n, [get_engine(d) for d in range(8)])
    sv.run(gl.from_circuit(circ), [])
    s = math.sin(theta / 2) ** 2
    levels = [(n - 2 * j, math.comb(n, j), s**j * (1 - s) ** (n - j)) for j in range(n, -1, -1)]  # ascending energy
    p_max = max(p for _, _, p in levels)
    for alpha in (0.05, 0.5, 0.9):
        value, _ = sv.cvar([1 << q for q in range(n)], [1.0] * n, alpha)
        bound = alpha - (1e-8 + 1e-5 * alpha)
        acc = taken = 0.0
        for e, cnt, p in levels:
            take = min(cnt * p, bound - taken)
            acc, taken = acc + take * e, taken + take
            if taken >= bound:
                break
        want = acc / alpha
        assert abs(value - want) <= n * p_max / alpha + 1e-9 * n, (alpha, value, want)
    sv.close()
