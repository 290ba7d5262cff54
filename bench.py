#!/usr/bin/env python
"""Benchmark of the EVQE circuit-evaluation hot path (BASELINE.json: "EVQE circuit evals/sec at 20q; gate-apply
HBM GB/s vs peak; at 1/2/4/8 GPU").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--layers L] [--dump-outputs DIR]

Workload (BASELINE.json configs[1], SURVEY.md section 8d "C2"): a population of 32 random EVQE individuals
(reference generation rules, seed 0 on EVERY rank) on 20 qubits with L parameterised layers, evaluated against a
synthetic random diagonal Ising Hamiltonian (20 Z + 190 ZZ terms, default_rng(1234)) -- one "step" = one batched
``evaluate_circuits`` submission of the whole population, i.e. one EVQE selection pass.
  value     circuit evaluations / s with parameters + plans resident on the device (CUDA events, kernels only)
  e2e       the same through ``B200OperatorCircuitEvaluator.evaluate_circuits`` with host lists in / floats out
  roofline  algorithmic bytes (2 * 16 B * 2^n per swept statevector) / CUDA-event time of the sweep kernel
Extras on rank 0 at N = 1 (``--skip-extras`` drops them): ``gate_apply`` (sweep kernel on ONE 24/26/28/30-qubit state, whole
circuit incl. the write-only first sweep), ``cpu_baseline`` (C/OpenMP oracle port on the host cores), ``c3_24q_tfim``,
``c4_26q_sampler`` (BASELINE configs 3 and 4 through the evaluators, with the error against the C oracle), ``e2e_threaded``
(the reference's calling pattern: 32 threads x single-circuit calls), ``optimizer_calls`` (one circuit, one or two parameter points
per call, last layer parameterised: microseconds per call).
``--dump-outputs DIR`` writes what the timed paths returned in their last step as float64 ``DIR/<name>.npy`` (rank 0): the inputs
are seeded, so two builds run with the same arguments can be compared output for output.
Multi-GPU (torchrun, one process per GPU): the headline is WEAK scaling -- every rank evaluates the same population of 32, no
data-path collective.  Extras at N > 1: ``strong`` (ONE population of 32 split over the N ranks + an all-gather of the 32
doubles per step), ``api_all_devices`` (ONE process driving all N GPUs through ``B200EstimatorV2(devices="all")``, the
configuration a QUEASARS user has) and ``sharded`` (a (32 + log2 N)-qubit state -- 35 qubits on 8 GPUs, BASELINE config C5 --
with the fused peer-memory global-qubit swap, plus a 28-qubit sharded run checked against the single-GPU engine).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_QUBITS = 20
POPULATION = 32
METRIC = "evqe_circuit_evals_per_sec_20q"
UNIT = "circuit_evals/s"


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def profiled_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per sweep launch of this workload, from the committed ncu --set full
    capture (newest profiles/r*_sweep20_traffic.json); None when no capture is present."""
    import glob

    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_sweep20_traffic.json")), reverse=True):
        try:
            with open(path) as fh:
                return float(json.load(fh)["mean_traffic_bytes_per_launch"])
        except Exception:
            continue
    return None


class ClockSampler:
    """SM clock + throttle reasons of THIS rank's GPU during a timed region, sampled in-process through NVML (every rank
    samples its own device the same way: no helper process, no rank asymmetry)."""

    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}

    def __init__(self, device_index: int, enabled: bool = True, period_s: float = 0.004):
        self.device_index, self.enabled, self.period_s = device_index, enabled, period_s
        self.sm, self.reasons, self.smax = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        self._nvml = None

    def _physical_index(self) -> int:
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[self.device_index])
            except Exception:
                pass
        return self.device_index

    def _loop(self, handle):
        nv = self._nvml
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(handle, nv.NVML_CLOCK_SM)))
                mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(handle))
                for name, bit in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(self.period_s)

    def __enter__(self):
        if not self.enabled:
            return self
        try:
            import pynvml as nv

            nv.nvmlInit()
            self._nvml = nv
            handle = nv.nvmlDeviceGetHandleByIndex(self._physical_index())
            self.smax = float(nv.nvmlDeviceGetMaxClockInfo(handle, nv.NVML_CLOCK_SM))
            self._thread = threading.Thread(target=self._loop, args=(handle,), daemon=True)
            self._thread.start()
        except Exception:
            self._thread = None
        return self

    def __exit__(self, *exc):
        if self._thread is not None:
            self._stop.set()
            self._thread.join(timeout=2)

    def summary(self):
        if not self.enabled:
            return None
        if not self.sm:
            return self.smi_sample()
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.smax, "reasons": sorted(self.reasons), "samples": len(self.sm), "how": "NVML, in-process, this rank's GPU"}

    def smi_sample(self):
        """Fallback when NVML is not importable: one nvidia-smi query right after the timed region."""
        import subprocess

        query = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            out = subprocess.run(["nvidia-smi", f"--query-gpu={query}", "--format=csv,noheader,nounits", "-i", str(self._physical_index())],
                                 capture_output=True, text=True, timeout=10).stdout.strip().splitlines()[0]
            parts = [p.strip() for p in out.split(",")]
            reasons = [n for n, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]) if v.lower().startswith("active")]
            return {"sm_mhz": float(parts[1]), "sm_max_mhz": float(parts[2]), "reasons": sorted(reasons), "samples": 0, "how": "nvidia-smi, one query right after the timed region"}
        except Exception:
            return None


def build_workload(n_qubits: int, layers: int, population: int, seed: int):
    from queasars_b200 import genome as gn

    individuals = gn.random_population(n_qubits, layers, population, True, seed)
    circuits = [ind.to_circuit() for ind in individuals]
    params = [list(ind.parameter_values) for ind in individuals]
    return individuals, circuits, params


# ---------------------------------------------------------------------------------------------- CPU baseline
def circuit_instructions(circuit):
    instr = []
    for inst in circuit.data:
        ps = tuple(p.name if hasattr(p, "name") else float(p) for p in inst.operation.params)
        instr.append((inst.operation.name, tuple(q._index for q in inst.qubits), ps))
    return instr


def cpu_prepare(individuals):
    """Lower every individual to the C oracle's gate arrays (outside the timed region: conservative for the CPU arm,
    the reference re-transpiles and re-binds on every call)."""
    from oracle import c_oracle

    return [c_oracle.lower(circuit_instructions(ind.to_circuit()), list(ind.parameter_values)) for ind in individuals]


def cpu_evaluate(prepared, table, n_qubits):
    """Oracle port of the reference path on the host cores: simulate each individual with the C/OpenMP oracle
    (oracle/c/statevector.c: one OpenMP team of all host threads per gate, like a compiled CPU simulator), then <H> from
    the precomputed diagonal table (conservative: the reference's estimator evaluates 210 Pauli terms per call instead)."""
    from oracle import c_oracle

    lib = c_oracle.load()
    state = np.empty(1 << n_qubits, dtype=np.complex128)
    out = []
    for targets, controls, mats in prepared:
        out.append(float(lib.oracle_run_circuit(state.ctypes.data, n_qubits, len(targets), targets.ctypes.data, controls.ctypes.data, mats.ctypes.data, table.ctypes.data)))
    return out


def cpu_table(n_qubits):
    from oracle import c_oracle
    from queasars_b200 import genome as gn

    _, z, c = gn.ising_operator(n_qubits).masks()
    return c_oracle.diag_table(n_qubits, [(int(a), float(b.real)) for a, b in zip(z, c)])


def host_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def claim_host_threads() -> int:
    """torchrun exports OMP_NUM_THREADS=1 to every rank: ask OpenMP explicitly for all host cores this process may use and
    return what the runtime then really provides (omp_get_max_threads)."""
    from oracle import c_oracle

    c_oracle.set_threads(host_threads())
    return c_oracle.max_threads()


def run_reference(args):
    """--impl reference: the reference's own CPU implementation is Qiskit (not installable offline), so this arm
    times the oracle port of it on the host cores: each step = a bounded sample of the same workload.  Under torchrun rank 0
    alone runs it (with all host cores); the other ranks exit."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    threads = claim_host_threads()
    sample = POPULATION
    individuals, _, _ = build_workload(N_QUBITS, args.layers, POPULATION, 0)
    prepared = cpu_prepare(individuals[:sample])
    table = cpu_table(N_QUBITS)
    for _ in range(max(1, min(args.warmup, 1))):
        cpu_evaluate(prepared, table, N_QUBITS)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        last = cpu_evaluate(prepared, table, N_QUBITS)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"values": last})
    value = sample * args.steps / dt
    desc = (f"{sample} of the {POPULATION} individuals per step on rank 0, C/OpenMP oracle port, omp_get_max_threads() = {threads} per evaluation "
            f"({host_threads()} host cores available to the process), diagonal table prebuilt")
    line = {
        "impl": "reference",
        "metric": METRIC,
        "value": value,
        "unit": UNIT,
        "n_gpus": max(args.gpus, world),
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f64",
        "data": "synthetic",
        "config": workload_config(args, max(args.gpus, world)),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": desc},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def dump_outputs(directory, arrays):
    """One float64 ``<name>.npy`` per entry of ``arrays`` (written after the timed region)."""
    os.makedirs(directory, exist_ok=True)
    for name, arr in arrays.items():
        np.save(os.path.join(directory, f"{name}.npy"), np.asarray(arr, dtype=np.float64))


def workload_config(args, n_gpus):
    return {
        "workload": f"C2: EVQE population of {POPULATION} individuals x {args.layers} layers, {N_QUBITS}-qubit random diagonal Ising (210 terms), one selection pass per step",
        "n_qubits": N_QUBITS,
        "population_per_gpu": POPULATION,
        "layers": args.layers,
        "precision": "complex128",
        "parallelism": f"population-parallel x{n_gpus} (the same population of {POPULATION} on every GPU, seed 0, no collective)",
        "l2": "working set 32 x 16 MiB = 512 MiB per step > 126 MB L2; no explicit flush",
    }


# ---------------------------------------------------------------------------------------------- GPU arm
def run_b200(args):
    import torch

    # keep stdout clean for the single JSON line: libraries (e.g. NCCL's version banner) write to fd 1 during set-up
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        import datetime

        # a rank that fails inside a collective section must not keep the others waiting for NCCL's default ten minutes
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(seconds=120))

    from queasars_b200 import B200EstimatorV2, B200OperatorCircuitEvaluator
    from queasars_b200 import genome as gn

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # the SAME population on every rank: the weak-scaling curve then measures the hardware, not population differences
    individuals, circuits, params = build_workload(N_QUBITS, args.layers, POPULATION, 0)
    operator = gn.ising_operator(N_QUBITS)
    estimator = B200EstimatorV2(device=local_rank, dtype="complex128", coalesce=False)
    evaluator = B200OperatorCircuitEvaluator(estimator, 0.0, operator)
    engine = estimator.engine
    values = evaluator.evaluate_circuits(circuits, params)  # compiles plans, builds the table
    assert len(values) == POPULATION and all(np.isfinite(values))

    plans = [estimator._cache.plan_for(c, probabilities_only=True) for c in circuits]  # the plans the evaluator call above compiled (diagonal H)
    ham = estimator.hamiltonian_for(operator)
    batch = engine.resident_batch(plans, ham)
    h2d = batch.set_params(params)
    stream = torch.cuda.ExternalStream(engine.stream, device=torch.device("cuda", local_rank))
    warmup = max(3, args.warmup)
    for _ in range(warmup):
        batch.run()
    resident = batch.read()
    assert np.allclose(resident, values, rtol=0, atol=1e-12)

    # ---- value: device-resident throughput, CUDA events on the launching stream ----
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    launches0 = engine.launch_count
    with ClockSampler(local_rank) as clocks:
        ev0.record(stream)
        for _ in range(args.steps):
            batch.run()
        ev1.record(stream)
        engine.synchronize()
        torch.cuda.synchronize()
    gpu_launches = engine.launch_count - launches0
    barrier()
    last_values = batch.read()  # the last timed step's results (read after the events: not part of the timed region)
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    ms_per_step = ms_total / args.steps
    value = world * POPULATION * args.steps / (ms_total * 1e-3)
    clock_info = clocks.summary()
    if world > 1 and clock_info is not None:  # every rank sampled its own GPU: report the slowest median and all reasons seen
        gathered = [None] * world
        dist.all_gather_object(gathered, clock_info)
        ok = [g for g in gathered if g]
        clock_info = dict(clock_info, sm_mhz=min(g["sm_mhz"] for g in ok), reasons=sorted({r for g in ok for r in g["reasons"]}),
                          per_rank_sm_mhz=[g["sm_mhz"] for g in ok])

    # ---- e2e: public evaluator API, host lists in, floats out (H2D of parameters + D2H of results inside) ----
    for _ in range(warmup):
        evaluator.evaluate_circuits(circuits, params)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = evaluator.evaluate_circuits(circuits, params)
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e_value = world * POPULATION * args.steps / e2e_s
    assert np.allclose(out, values, rtol=0, atol=1e-12)
    if args.dump_outputs and rank == 0:
        # "values": device-resident batch (the headline), "e2e_values": B200OperatorCircuitEvaluator.evaluate_circuits
        dump_outputs(args.dump_outputs, {"values": last_values, "e2e_values": out})

    # ---- roofline of the dominant kernel (sweep_kernel<double>), live CUDA events ----
    peak, peak_kind = measured_peak_gbs()
    stats = batch.stats()
    sweep_bytes = stats["sweep_bytes"]
    # algorithmic bytes of one step: every read+write sweep moves 2 * 16 B * 2^n per state, the first sweep of a circuit
    # only writes (it synthesises the product-state start), the last sweep of a circuit only reads (the Hamiltonian is
    # diagonal: <H> is accumulated in the sweep's epilogue and the final state, which nothing reads, is not written back),
    # and that epilogue reads the 8 B * 2^n table once per circuit (SURVEY.md section 8d)
    tot_ms, tot_bytes = 0.0, 0.0
    for _ in range(3):
        ms, states = batch.run_timed()
        tot_ms += float(ms.sum())
        tot_bytes += float(sweep_bytes * (states.sum() - 0.5 * states[0] - 0.5 * POPULATION) + POPULATION * 8 * (1 << N_QUBITS))
    step_bytes = tot_bytes / 3
    # The sweep launches of a step overlap (two stream groups), so "one launch's duration" is not what a step pays: the achieved
    # figure is the step's algorithmic sweep bytes over the CUDA-event time of the timed region (the sweep kernel is 98 % of the
    # device time: profiles/r2_bench_launches_summary.txt; taking the whole step is the conservative choice).  The same kernel
    # timed launch by launch on ONE stream (run_timed: event pair around every launch, no overlap) is reported beside it.
    achieved = step_bytes / (ms_per_step * 1e-3) / 1e9
    serialized = tot_bytes / (tot_ms * 1e-3) / 1e9
    # FP64 side of the roofline: DFMA-class instructions the applied gates need, counted from the plans' own ops (after the
    # front end's rewrites), against the sustained DFMA issue rate measured on this pool's B200 (tools/fp64_peak.cu).
    from queasars_b200 import gate_list as _gl
    from queasars_b200 import schedule as _sc

    dfma = 0.0
    from queasars_b200 import engine as _eng

    for c in circuits:
        ops = _eng.rewritten(estimator._cache.gates_for(c)["gates"], drop_final_phases=True).ops
        _, remaining = _sc.split_product_prefix(ops, N_QUBITS)
        dfma += sum(_gl.dfma_per_amplitude(ops[i]) for i in remaining) * float(1 << N_QUBITS)
    fp64_peak = 16.9e12
    fp64_rate = dfma / (ms_per_step * 1e-3)
    n_plan_ops = float(np.mean([p.n_ops for p in plans]))
    roofline = {
        "bound": "hbm",
        "kernel": "qb::sweep_kernel<double>",
        "achieved": achieved,
        "peak": peak,
        "peak_kind": peak_kind,
        "unit": "GB/s",
        "frac": achieved / peak,
        "traffic": profiled_traffic(),
        "algorithmic_bytes_per_step": step_bytes,
        "algorithmic_bytes_per_launch": step_bytes / max(1, stats["sweep_launches"]),
        "serialized_launches": {"GBps": serialized, "frac": serialized / peak, "ms_per_step": tot_ms / 3,
                                "how": "event pair around every sweep launch on one stream (no overlap between launches)"},
        "bytes_per_statevector_sweep": sweep_bytes,
        "sweeps_per_evaluation": stats["state_sweeps"] / POPULATION,
        "gates_per_sweep": n_plan_ops / (stats["state_sweeps"] / POPULATION),
        "sweep_share_of_step": 0.98,
        "fp64": {"dfma_instr_per_s": fp64_rate, "peak_measured": fp64_peak, "frac": fp64_rate / fp64_peak, "unit": "DFMA-class instr/s"},
        "note": "sweeps of this workload fuse ~16 applied fp64 gates each: the binding roof is FP64 issue (see fp64), not HBM; gate_apply reports the HBM-bound regime at 24-30 q",
    }

    line = {
        "metric": METRIC,
        "value": value,
        "unit": UNIT,
        "n_gpus": world,
        "steps": args.steps,
        "warmup": warmup,
        "ms_per_step": ms_per_step,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f64",
        "data": "synthetic",
        "config": workload_config(args, world),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 8 * POPULATION, "ms_per_step": 1e3 * e2e_s / args.steps},
        "gpu_launches": int(gpu_launches),
        "roofline": roofline,
        "clocks": clock_info,
    }

    if not args.skip_extras:
        if world == 1:
            line["gate_apply"] = guarded(lambda: gate_apply_probe(engine, peak))
            line["cpu_baseline"] = guarded(lambda: cpu_baseline_leg(individuals, values))
            line["c3_24q_tfim"] = guarded(lambda: c3_probe(local_rank))
            line["c4_26q_sampler"] = guarded(lambda: c4_probe(local_rank))
            line["e2e_threaded"] = guarded(lambda: threaded_probe(local_rank, operator, circuits, params, values, args))
            line["optimizer_calls"] = guarded(lambda: optimizer_calls_probe(local_rank, operator, individuals))
            line["c1_jssp_reference_loop"] = guarded(lambda: c1_probe(local_rank))
            line["c2_complex64"] = guarded(lambda: complex64_probe(local_rank, operator, circuits, params, values, args))
        else:
            line["strong"] = guarded(lambda: strong_probe(dist, rank, world, engine, plans, ham, params, values, args, barrier, max_over_ranks))
            batch.close()
            line["api_all_devices"] = guarded(lambda: all_devices_probe(dist, rank, world, operator, circuits, params, values, args))
            torch.cuda.set_device(local_rank)
            line["sharded"] = guarded(lambda: sharded_probe(dist, rank, world, local_rank))
    if world > 1:
        dist.destroy_process_group()
    sys.stdout.flush()
    os.dup2(json_fd, 1)
    os.close(json_fd)
    if rank == 0:
        print(json.dumps(line), flush=True)


def guarded(fn):
    """An extra must never cost the headline line: failures are reported in place."""
    try:
        return fn()
    except Exception as exc:  # noqa: BLE001
        return {"error": f"{type(exc).__name__}: {exc}"}


# ---------------------------------------------------------------------------------------------- extras, N = 1
def gate_apply_probe(engine, peak, sizes=((24, 6), (26, 6), (28, 4), (30, 4))):
    """The sweep kernel on ONE HBM-resident state of 24 / 26 / 28 / 30 qubits (0.25 / 1 / 4 / 16 GiB), two circuits each:
      fused_evqe   a random EVQE individual: ~20 gates fused per sweep -> FP64-issue bound by design
      hbm_regime   3 layers of 7 ``u`` gates on 7 non-low qubits behind a product start -> HBM and FP64 time about equal
      hbm_sparse   3 layers of 3 such gates -> HBM bound
    Reported for the WHOLE circuit, first (write-only, product-state) sweep included: algorithmic bytes = 16 B * 2^n for the
    first sweep + 2 * 16 B * 2^n for every later one, divided by the CUDA-event time of all sweep launches; ``rw_sweeps``
    repeats the figure for the read+write sweeps alone.  ``gates_in_sweeps`` = ops the plan really put into each sweep."""
    from queasars_b200 import engine as eng_mod
    from queasars_b200 import gate_list as gl
    from queasars_b200 import genome as gn
    from queasars_b200.circuit import QuantumCircuit

    def measure(gates, params, reps):
        # planned like the evaluators plan for a diagonal observable / sampling (engine.rewritten: trailing phases deferred)
        plan = engine.compile(gates, drop_final_phases=True)
        _, _, _, (sweeps, _, _, _, _) = eng_mod.encoded_plan(eng_mod.rewritten(gates, True), engine.tile_bits, engine.reg_bits, True)
        rb = engine.resident_batch([plan], None)
        rb.set_params([params])
        for _ in range(2):
            rb.run()
        per_sweep = np.zeros(plan.n_sweeps)
        for _ in range(reps):
            ms, _states = rb.run_timed()
            per_sweep += ms
        per_sweep /= reps
        half = rb.stats()["sweep_bytes"] / 2  # 16 B * 2^n
        rb.close()
        total_ms = float(per_sweep.sum())
        bytes_all = half * (2 * plan.n_sweeps - 1)
        out = {
            "sweeps": int(plan.n_sweeps),
            "gates_in_sweeps": [int(s["op_end"] - s["op_begin"]) for s in sweeps],
            "ms_per_sweep": [round(float(v), 4) for v in per_sweep],
            "ms_per_circuit": total_ms,
            "GBps_whole_circuit": bytes_all / (total_ms * 1e-3) / 1e9,
        }
        out["frac_of_measured_hbm"] = out["GBps_whole_circuit"] / peak
        if plan.n_sweeps > 1:
            rw_ms = float(per_sweep[1:].sum())
            out["rw_sweeps"] = {"GBps": 2 * half * (plan.n_sweeps - 1) / (rw_ms * 1e-3) / 1e9}
            out["rw_sweeps"]["frac_of_measured_hbm"] = out["rw_sweeps"]["GBps"] / peak
            out["first_sweep_write_only_GBps"] = half / (float(per_sweep[0]) * 1e-3) / 1e9
        return out

    result = {}
    for n, layers in sizes:
        ind = gn.Individual.random(n, layers, True, 7)
        fused = measure(gl.from_evqe_individual(ind), list(ind.parameter_values), 3)
        fused["layers"] = layers
        circ = QuantumCircuit(n)
        for q in range(n):
            circ.u(0.1 + 0.01 * q, 0.2, 0.3, q)  # absorbed into the product-state start
        for layer in range(3):
            for g in range(7):
                circ.u(0.3 + g, 0.2 * layer, 0.1, 4 + ((g * 3 + 7 * layer) % (n - 4)))
        hbm = measure(gl.from_circuit(circ), [], 3)
        # the same with 3 gates per layer: at 7 gates a sweep's FP64 work already takes as long as its HBM traffic (the write-only
        # first sweep is as slow as the read+write ones), at 3 the traffic alone is left
        sparse_circ = QuantumCircuit(n)
        for q in range(n):
            sparse_circ.u(0.1 + 0.01 * q, 0.2, 0.3, q)
        for layer in range(3):
            for g in range(3):
                sparse_circ.u(0.3 + g, 0.2 * layer, 0.1, 4 + ((g * 5 + 3 * layer) % (n - 4)))
        sparse = measure(gl.from_circuit(sparse_circ), [], 3)
        result[f"{n}q"] = {"fused_evqe": fused, "hbm_regime": hbm, "hbm_sparse": sparse}
    return result


def cpu_baseline_leg(individuals, gpu_values):
    threads = claim_host_threads()
    sample = len(individuals)
    table = cpu_table(N_QUBITS)
    prepared = cpu_prepare(individuals[:sample])
    t0 = time.perf_counter()
    vals = cpu_evaluate(prepared, table, N_QUBITS)
    reps = 1
    while time.perf_counter() - t0 < 10.0 and reps < 8:
        cpu_evaluate(prepared, table, N_QUBITS)
        reps += 1
    dt = time.perf_counter() - t0
    err = float(np.max(np.abs(np.asarray(vals) - np.asarray(gpu_values[:sample])) / np.maximum(1.0, np.abs(vals))))
    return {
        "value": sample * reps / dt,
        "unit": UNIT,
        "cores": threads,
        "kind": "port",
        "sample": f"{reps} x {sample} of the {POPULATION} individuals, C/OpenMP oracle port of the Qiskit statevector estimator (omp_get_max_threads() = {threads} per evaluation), diagonal table prebuilt",
        "max_rel_err_gpu_vs_oracle": err,
    }


def c3_probe(device):
    """BASELINE config 3: 24-qubit open-chain transverse-field Ising Pauli sum (23 ZZ + 24 X), fp64, 4 random EVQE individuals
    of 6 layers per ``evaluate_circuits`` call; error of every value against the C oracle (one pass per Pauli term)."""
    from oracle import c_oracle
    from queasars_b200 import B200EstimatorV2, B200OperatorCircuitEvaluator
    from queasars_b200 import genome as gn

    n, batch = 24, 4
    pop = gn.random_population(n, 6, batch, True, 0)
    circuits, params = [i.to_circuit() for i in pop], [list(i.parameter_values) for i in pop]
    op = gn.tfim_operator(n)
    ev = B200OperatorCircuitEvaluator(B200EstimatorV2(device=device, coalesce=False), 0.0, op)
    vals = ev.evaluate_circuits(circuits, params)
    reps = 10
    t0 = time.perf_counter()
    for _ in range(reps):
        vals = ev.evaluate_circuits(circuits, params)
    dt = (time.perf_counter() - t0) / reps
    claim_host_threads()
    terms = op.to_list()
    state = np.empty(1 << n, dtype=np.complex128)
    err, t_cpu = 0.0, 0.0
    for ind, circ, v in zip(pop[:2], circuits, vals):
        t1 = time.perf_counter()
        c_oracle.evaluate(circuit_instructions(circ), n, list(ind.parameter_values), None, state)
        want = c_oracle.pauli_sum(state, n, terms)
        t_cpu += time.perf_counter() - t1
        err = max(err, abs(v - want) / max(1.0, abs(want)))
    return {"workload": f"{batch} individuals x 6 layers per call, 47 Pauli terms", "evals_per_s": batch / dt, "ms_per_call": 1e3 * dt,
            "max_rel_err_vs_c_oracle": err, "checked": 2, "cpu_oracle_evals_per_s": 2 / t_cpu}


def c4_probe(device):
    """BASELINE config 4: 26-qubit JSSP QUBO (3 jobs / 5 machines, 84 distinct diagonal terms), 10 000 shots per individual,
    4 random EVQE individuals of 4 layers per call through the sampler evaluator (alpha = 1 and CVaR 0.5); the sampled
    indices of one individual are compared with the C oracle's cumsum -> searchsorted(right) on the same uniforms."""
    from oracle import c_oracle
    from queasars_b200 import B200OperatorSamplerCircuitEvaluator, B200SamplerV2
    from queasars_b200 import genome as gn
    from queasars_b200.operators import SparsePauliOp

    golden = json.load(open(os.path.join(ROOT, "tests", "golden", "jssp_hamiltonians.json")))["jssp_26q"]
    n, batch, shots, seed = 26, 4, 10000, 3
    op = SparsePauliOp._raw(n, [0] * golden["n_raw_terms"], golden["z_masks"], golden["coeffs"])
    pop = gn.random_population(n, 4, batch, True, 1)
    circuits, params = [i.to_circuit() for i in pop], [list(i.parameter_values) for i in pop]
    out = {"workload": f"{batch} individuals x 4 layers per call, {shots} shots each"}
    sampler = B200SamplerV2(device=device, seed=seed, coalesce=False)
    for alpha in (1.0, 0.5):
        ev = B200OperatorSamplerCircuitEvaluator(sampler, shots, op, alpha=alpha)
        ev.evaluate_circuits(circuits, params)
        reps = 3
        t0 = time.perf_counter()
        for _ in range(reps):
            vals = ev.evaluate_circuits(circuits, params)
        dt = (time.perf_counter() - t0) / reps
        out[f"alpha_{alpha}"] = {"evals_per_s": batch / dt, "ms_per_call": 1e3 * dt, "values": [float(v) for v in vals[:2]]}
    claim_host_threads()
    state = np.empty(1 << n, dtype=np.complex128)
    c_oracle.evaluate(circuit_instructions(circuits[0]), n, params[0], None, state)
    uniforms = np.random.default_rng(seed).random(shots)
    want = c_oracle.sample_indices(state, n, uniforms)
    got = sampler.sample_indices([circuits[0]], [params[0]], shots)[0]
    flips = np.nonzero(got != want)[0]
    probs = state.real**2 + state.imag**2
    out["index_mismatches_vs_c_oracle"] = int(flips.size)
    # a mismatch is a uniform within rounding of a CDF boundary (the GPU sums |psi|^2 in 512-amplitude chunks, the oracle
    # sequentially): the two draws must then be CDF neighbours -- the probability mass strictly between them is below the
    # rounding of a 2^26-term sum
    between = [float(np.sum(probs[min(int(got[i]), int(want[i])) + 1 : max(int(got[i]), int(want[i]))])) for i in flips]
    out["max_probability_mass_between_mismatched_draws"] = max(between) if between else 0.0
    out["mismatches_are_cdf_neighbours"] = bool(all(m < 1e-10 for m in between) and all(probs[got[i]] > 0 for i in flips))
    out["shots_checked"] = shots
    return out


def c1_probe(device):
    """BASELINE config 1: the reference's OWN ``EVQEMinimumEigensolver`` loop (unmodified package from the git-ignored
    ``baseline/_ref``, staged by tools/stage_reference.py) on the small JSSP instances of its example notebooks, sampler-only
    CVaR(0.5) objective as in examples/evqe_jssp_small_examples.ipynb cell 10, with ``B200SamplerV2`` handed to it inside
    ``ConfiguredSamplerV2``.  Reports the objective reached (notebook values: 63.5 / 61.6 / 22.75), the circuit evaluations the
    loop spent and its wall time (the loop itself -- Python threads, SPSA, genome operators -- is the reference's)."""
    from concurrent.futures import ThreadPoolExecutor

    ref_path = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isfile(os.path.join(ref_path, "queasars", "__init__.py")):
        return {"skipped": "baseline/_ref not staged (python tools/stage_reference.py in the build container)"}
    from queasars_b200 import B200SamplerV2
    from tests import reference_loop

    ref = reference_loop.import_reference(ref_path)
    out = {}
    for which in ("4q", "5q", "8q"):
        _, hamiltonian, best = reference_loop.jssp_instance(ref, which)
        sampler = B200SamplerV2(device=device, seed=7)
        with ThreadPoolExecutor(max_workers=10) as pool:
            solver = reference_loop.jssp_solver(ref, sampler, pool, random_seed=0)
            t0 = time.perf_counter()
            result = solver.compute_minimum_eigenvalue(operator=hamiltonian)
            dt = time.perf_counter() - t0
        evals = int(sum(result.circuit_evaluations))
        out[which] = {"objective": float(result.eigenvalue), "notebook_value": best, "circuit_evaluations": evals, "seconds": dt, "evals_per_s": evals / dt,
                      "generations": len(result.circuit_evaluations)}
    return out


def complex64_probe(device, operator, circuits, params, values, args):
    """The optional complex64 path on the headline workload (same population, same Hamiltonian): end-to-end evals/s through the
    evaluator and the error against the complex128 values (north star: 1e-4 relative in fp32).  Not the headline: BASELINE's metric
    is complex128."""
    from queasars_b200 import B200EstimatorV2, B200OperatorCircuitEvaluator

    est = B200EstimatorV2(device=device, dtype="complex64", coalesce=False)
    ev = B200OperatorCircuitEvaluator(est, 0.0, operator)
    got = ev.evaluate_circuits(circuits, params)
    err = float(np.max(np.abs(np.asarray(got) - np.asarray(values)) / np.maximum(1.0, np.abs(values))))
    reps = max(10, min(args.steps, 100))
    t0 = time.perf_counter()
    for _ in range(reps):
        ev.evaluate_circuits(circuits, params)
    dt = time.perf_counter() - t0
    return {"evals_per_s": POPULATION * reps / dt, "ms_per_call": 1e3 * dt / reps, "max_rel_err_vs_complex128": err, "tolerance": 1e-4}


def optimizer_calls_probe(device, operator, individuals):
    """The optimizer loop's calling pattern (mutation.py:59-77: SPSA / NFT evaluate ONE circuit with only its last layer
    parameterised at one or two points per call, sequentially): microseconds per call through the evaluator
    (``evaluate_circuits([circuit] * k, rows)``, prefix-state reuse and the cached CUDA graph behind it) and at the engine level,
    for the last-layer circuit and for the fully parameterised one.  20 qubits, the headline Hamiltonian."""
    from queasars_b200 import B200EstimatorV2, B200OperatorCircuitEvaluator
    from queasars_b200 import gate_list as gl

    ind = individuals[0]
    est = B200EstimatorV2(device=device, dtype="complex128", coalesce=False)
    ev = B200OperatorCircuitEvaluator(est, 0.0, operator)
    engine = est.engines[0] if hasattr(est, "engines") else est.engine
    ham = engine.hamiltonian(operator)
    rng = np.random.default_rng(5)
    out = {"n_qubits": ind.n_qubits, "layers": len(ind.layers)}
    for name, layers in (("last_layer", {-1}), ("all_layers", None)):
        circuit = ind.to_circuit(layers)
        gates = gl.from_evqe_individual(ind, layers)
        plan = engine.compile_with_prefix_reuse(gates, drop_final_phases=True) if layers else engine.compile(gates, drop_final_phases=True)
        for points in (1, 2):
            rows = [list(rng.uniform(0, 6.28, gates.n_params)) for _ in range(points)]
            res = {}
            for label, call in (("evaluator_us_per_call", lambda: ev.evaluate_circuits([circuit] * points, rows)),
                                ("engine_us_per_call", lambda: engine.expectation([plan] * points, rows, ham))):
                for _ in range(30):
                    call()
                reps = 500
                t0 = time.perf_counter()
                for _ in range(reps):
                    call()
                res[label] = 1e6 * (time.perf_counter() - t0) / reps
            want = engine.expectation([plan] * points, rows, ham)
            res["evaluator_matches_engine"] = bool(np.allclose(ev.evaluate_circuits([circuit] * points, rows), want, rtol=0, atol=1e-12))
            out[f"{name}_{points}pt"] = res
    return out


def threaded_probe(device, operator, circuits, params, values, args):
    """The reference's own calling pattern (selection.py:75-82, evqe.py:232-236): ``population_size`` threads, each submitting
    single-circuit ``evaluate_circuits`` calls, coalesced by the sleep-free batching queue (coalesce=True)."""
    from concurrent.futures import ThreadPoolExecutor

    from queasars_b200 import B200EstimatorV2, B200OperatorCircuitEvaluator

    est = B200EstimatorV2(device=device, dtype="complex128", coalesce=True)
    ev = B200OperatorCircuitEvaluator(est, 0.0, operator)
    rounds = max(10, min(args.steps, 100))

    def work(i):
        last = None
        for _ in range(rounds):
            last = ev.evaluate_circuits([circuits[i]], [params[i]])[0]
        return last

    rates = []
    with ThreadPoolExecutor(max_workers=POPULATION) as pool:
        list(pool.map(work, range(POPULATION)))  # warm-up: plans, table, thread start
        for _ in range(5):  # thread scheduling makes single runs scatter: median of five, range reported
            t0 = time.perf_counter()
            got = list(pool.map(work, range(POPULATION)))
            rates.append(POPULATION * rounds / (time.perf_counter() - t0))
    assert np.allclose(got, values, rtol=0, atol=1e-12)
    q = est._queue
    return {"evals_per_s": float(np.median(rates)), "min": float(min(rates)), "max": float(max(rates)), "runs": len(rates), "threads": POPULATION,
            "calls_per_thread": rounds, "mean_coalesced_batch": q.requests_executed / max(1, q.batches_executed),
            "pattern": "32 threads x single-circuit evaluate_circuits calls, coalesce=True"}


# ---------------------------------------------------------------------------------------------- extras, N > 1
def strong_probe(dist, rank, world, engine, plans, ham, params, values, args, barrier, max_over_ranks):
    """STRONG scaling: ONE population of 32 split over the N ranks (longest-processing-time by sweep count, the same split on
    every rank), each step = evaluate the share + all-gather of the 32 doubles so that every rank holds the whole
    generation's values (what EVQE's selection needs: selection.py:75-88).  Wall clock around K steps, max over ranks."""
    import torch

    order = sorted(range(POPULATION), key=lambda i: (-plans[i].n_sweeps, -plans[i].n_ops, i))
    load, owner = [0.0] * world, [0] * POPULATION
    for i in order:
        r = min(range(world), key=lambda d: (load[d], d))
        owner[i] = r
        load[r] += plans[i].n_sweeps * 1000 + plans[i].n_ops
    mine = [i for i in range(POPULATION) if owner[i] == rank]
    counts = [owner.count(r) for r in range(world)]
    width = max(counts)
    batch = engine.resident_batch([plans[i] for i in mine], ham) if mine else None
    if batch is not None:
        batch.set_params([params[i] for i in mine])
    send = torch.zeros(width, dtype=torch.float64, device="cuda")
    recv = torch.zeros(world * width, dtype=torch.float64, device="cuda")

    def step():
        if batch is not None:
            batch.run()
            send[: len(mine)] = torch.from_numpy(batch.read()).cuda()
        dist.all_gather_into_tensor(recv, send)
        return recv

    for _ in range(3):
        step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        got = step()
    torch.cuda.synchronize()
    dt = max_over_ranks(time.perf_counter() - t0)
    gathered = got.cpu().numpy().reshape(world, width)
    full = np.empty(POPULATION)
    for r in range(world):
        full[[i for i in range(POPULATION) if owner[i] == r]] = gathered[r, : counts[r]]
    assert np.allclose(full, values, rtol=0, atol=1e-12)
    if batch is not None:
        batch.close()
    return {"value": POPULATION * args.steps / dt, "unit": UNIT, "scaling": "strong", "ms_per_step": 1e3 * dt / args.steps,
            "individuals_per_rank": counts, "collective": f"all_gather_into_tensor of {world} x {width} doubles per step (NCCL)",
            "note": "one population of 32 over all ranks; compare with the N=1 e2e value for strong-scaling efficiency"}


def all_devices_probe(dist, rank, world, operator, circuits, params, values, args):
    """ONE process, ALL GPUs, through the drop-in API: ``B200EstimatorV2(devices="all")`` behind
    ``B200OperatorCircuitEvaluator.evaluate_circuits`` -- the configuration a QUEASARS user has (ThreadPoolExecutor around one
    primitive: evqe.py:232-236).  Rank 0 runs it while the other ranks wait at a barrier with idle GPUs."""
    import torch

    # the other ranks must wait on the CPU: an NCCL barrier is a kernel spinning on their GPU, i.e. on the GPUs rank 0 is about to use
    cpu_group = dist.new_group(backend="gloo")
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    out, error = None, None
    if rank == 0:
        try:
            out = _all_devices_rank0(operator, circuits, params, values, args)
        except Exception as exc:  # noqa: BLE001 -- the waiting ranks must be released whatever happens here
            error = exc
    dist.barrier(group=cpu_group)  # gloo: the waiting ranks sleep on a socket, their GPUs stay idle
    if error is not None:
        raise error
    return out


def _all_devices_rank0(operator, circuits, params, values, args):
    from queasars_b200 import B200EstimatorV2, B200OperatorCircuitEvaluator

    est = B200EstimatorV2(devices="all", dtype="complex128", coalesce=False)
    ev = B200OperatorCircuitEvaluator(est, 0.0, operator)
    for _ in range(3):
        got = ev.evaluate_circuits(circuits, params)
    assert np.allclose(got, values, rtol=0, atol=1e-12)
    before = [e.launch_count for e in est.engines]
    steps = max(10, args.steps)
    t0 = time.perf_counter()
    for _ in range(steps):
        got = ev.evaluate_circuits(circuits, params)
    dt = time.perf_counter() - t0
    used = [e.launch_count - b for e, b in zip(est.engines, before)]
    return {"value": POPULATION * steps / dt, "unit": UNIT, "ms_per_call": 1e3 * dt / steps, "devices": est.devices_used(),
            "kernel_launches_per_device": used, "pattern": "one evaluate_circuits call of 32 circuits per step, one process, one worker thread per GPU"}


def sharded_probe(dist, rank, world, local_rank):
    """BASELINE config C5 at this N: ONE (32 + log2 N)-qubit complex128 statevector (35 qubits = 512 GiB on 8 GPUs, 2 x 64 GiB
    ping-pong buffers per GPU) sharded by its top qubits, a product-state circuit whose second half forces one global-qubit
    swap, checked against the closed forms of <Z>, <ZZ> and the transverse-field Ising sum; swap time and NVLink GB/s per
    direction per GPU.  Before it, a 28-qubit random EVQE individual on the same ranks is compared with the single-GPU engine."""
    import torch

    from queasars_b200 import gate_list as gl
    from queasars_b200 import genome as gn
    from queasars_b200.circuit import QuantumCircuit
    from queasars_b200.operators import SparsePauliOp
    from queasars_b200.sharded import ShardedStatevector

    g = int(round(math.log2(world)))
    out = {}

    def diag_terms(n):
        _, z, c = gn.ising_operator(n, seed=3).masks()
        return z[: 2 * n], c.real[: 2 * n]

    # ---- 28 qubits, sharded vs single GPU
    n = 28
    ind = gn.Individual.random(n, 2, True, 11)
    gates = gl.from_evqe_individual(ind)
    z, c = diag_terms(n)
    sv = ShardedStatevector(n)
    sv.run(gates, ind.parameter_values)
    value = sv.diagonal_expectation(z, c)
    tf = sv.expectation(gn.tfim_operator(n))
    entry = {"n_qubits": n, "swaps": sv.swaps_done, "swap_path": "p2p kernel (peer memory)" if sv._peer_ptrs is not None else "nccl all_to_all",
             "swap_fallback_reason": getattr(sv, "swap_fallback_reason", None)}
    sv.close()  # collective: unmap the peers' buffers before anyone frees its own
    del sv
    torch.cuda.empty_cache()
    if rank == 0:
        from queasars_b200.primitives import get_engine

        eng = get_engine(local_rank, "complex128")
        plan = eng.compile(gates)
        ref = eng.expectation([plan], [list(ind.parameter_values)], eng.hamiltonian(SparsePauliOp._raw(n, [0] * len(z), [int(v) for v in z], [float(v) for v in c]), build_table=False))[0]
        tref = eng.expectation([plan], [list(ind.parameter_values)], eng.hamiltonian(gn.tfim_operator(n)))[0]
        entry.update(diag_rel_err_vs_single_gpu=abs(value - ref) / max(1.0, abs(ref)), tfim_rel_err_vs_single_gpu=abs(tf - tref) / max(1.0, abs(tref)))
    out["evqe_28q_vs_single_gpu"] = entry
    dist.barrier()

    # ---- (32 + g) qubits: as large as the free memory allows (two shard-sized buffers per GPU)
    free_b, _ = torch.cuda.mem_get_info()
    free_min = torch.tensor([free_b], dtype=torch.int64, device="cuda")
    dist.all_reduce(free_min, op=dist.ReduceOp.MIN)
    n_local = min(32, int(math.floor(math.log2(max(1, int(free_min.item()) * 0.85 / 32)))))
    n = n_local + g
    thetas = np.random.default_rng(5).uniform(0, np.pi, n)
    circ = QuantumCircuit(n)
    for _rep in range(2):  # two half rotations per qubit: the second one is a real gate on an existing state (and needs a swap)
        for q in range(n):
            circ.ry(float(thetas[q]) / 2, q)
    gates = gl.from_circuit(circ)
    z, c = diag_terms(n)
    cosines = np.cos(thetas)
    want = float(sum(cf * np.prod([cosines[q] for q in range(n) if (int(zm) >> q) & 1]) for zm, cf in zip(z, c)))
    want_tfim = float(-np.sum(np.cos(thetas[:-1]) * np.cos(thetas[1:])) - 0.5 * np.sum(np.sin(thetas)))
    sv = ShardedStatevector(n)
    torch.cuda.synchronize()
    dist.barrier()
    t0 = time.perf_counter()
    sv.run(gates, ())
    torch.cuda.synchronize()
    t_run = time.perf_counter() - t0
    swaps_in_run = sv.swaps_done
    value = sv.diagonal_expectation(z, c)
    norm = sv.norm_squared()
    t0 = time.perf_counter()
    tf = sv.expectation(gn.tfim_operator(n))
    t_tfim = time.perf_counter() - t0
    t0 = time.perf_counter()
    shots = sv.sample(10000, seed=123)
    t_sample = time.perf_counter() - t0
    marg = np.array([np.mean((shots >> q) & 1) for q in range(n)])
    lp = list(range(sv.n_local - sv.n_global, sv.n_local))
    for _ in range(2):
        sv._swap_all_global(lp)
    torch.cuda.synchronize()
    dist.barrier()
    t0 = time.perf_counter()
    reps = 4
    for _ in range(reps):
        sv._swap_all_global(lp)
    torch.cuda.synchronize()
    swap_ms = 1e3 * (time.perf_counter() - t0) / reps
    sent = 16 * (1 << sv.n_local) * (world - 1) / world
    out["c5"] = {
        "n_qubits": n, "n_local": sv.n_local, "state_GiB": 16 * (1 << n) / 2**30, "gates": len(gates.ops), "swaps_in_circuit": swaps_in_run, "circuit_s": t_run,
        "diag_rel_err_vs_closed_form": abs(value - want) / max(1.0, abs(want)), "tfim_rel_err_vs_closed_form": abs(tf - want_tfim) / max(1.0, abs(want_tfim)),
        "tfim_s": t_tfim, "norm_err": abs(norm - 1.0), "sample_10k_s": t_sample,
        "max_marginal_dev_sigma": float(np.max(np.abs(marg - np.sin(thetas / 2) ** 2)) / (0.5 / math.sqrt(len(shots)))),
        "swap_ms": swap_ms, "swap_sent_GB_per_gpu": sent / 1e9, "swap_GBps_per_direction_per_gpu": sent / (swap_ms * 1e-3) / 1e9,
        "swap_frac_of_nvlink5_900GBps": sent / (swap_ms * 1e-3) / 1e9 / 900.0,
        "swap_path": "swap_p2p_kernel: one fused kernel (peer stores over NVLink) + barrier" if sv._peer_ptrs is not None else "pack + all_to_all_single + unpack",
        "swap_fallback_reason": getattr(sv, "swap_fallback_reason", None),
    }
    sv.close()
    del sv
    torch.cuda.empty_cache()
    return out


def positive_int(text):
    value = int(text)
    if value < 1:
        raise argparse.ArgumentTypeError(f"must be at least 1, got {value}")
    return value


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=200,
                    help="timed steps of the headline and e2e loops (the e2e_threaded and complex64 legs clamp it to 10..100, api_all_devices to >= 10)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--layers", type=int, default=6)
    ap.add_argument("--skip-extras", action="store_true", help="headline line only: no gate-apply / C3 / C4 / threaded / CPU legs (N = 1), no strong / all-devices / sharded legs (N > 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results as float64 DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
