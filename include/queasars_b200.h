/*
 * queasars_b200 -- C-ABI of the B200 (sm_100a) statevector evaluation engine behind QUEASARS' EVQE loop.
 *
 * Plain C, plain pointers and sizes, no torch / C++ types.  The reference (DLR-RB/QUEASARS v0.3.2) is pure
 * Python and delegates this whole path to a Qiskit Estimator/Sampler primitive, so there is no existing
 * FFI; each entry point below names the reference interface whose work it takes over.  Paths are relative
 * to the reference checkout; [upstream] marks behaviour of un-vendored qiskit 2.4.2.
 *
 * Conventions
 *   - little-endian qubits: qubit q is bit q of the amplitude index (utility/pauli_strings.py:38-41)
 *   - statevectors are interleaved (re, im) complex128 (QB_C128) or complex64 (QB_C64)
 *   - every function returns QB_OK (0) or a negative error code; qb_last_error() gives the message of the
 *     last failure on the calling thread.  Nothing falls back to the CPU: without a CUDA device the
 *     compute entry points fail with QB_ERR_CUDA.
 *   - host buffers are owned by the caller and may be pageable; entry points are thread-safe per context.
 */
#ifndef QUEASARS_B200_H
#define QUEASARS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QB_OK 0
#define QB_ERR_INVALID (-1)
#define QB_ERR_CUDA (-2)
#define QB_ERR_MEMORY (-3)
#define QB_ERR_NOT_FOUND (-4)

#define QB_C128 0
#define QB_C64 1

#define QB_TILE_BITS 11     /* default amplitudes per CTA tile = 2^11 (a plan may choose 12) */
#define QB_MAX_TILE_BITS 12
#define QB_REG_BITS 4   /* default amplitudes per thread = 2^4 (a plan may choose 3 with 2^11 tiles: 32 warps / SM, measured slower) */
#define QB_LOW_BITS 4   /* lowest qubits always inside the tile (256 B contiguous runs for c128) */

/* operand-position kinds inside a pass (see queasars_b200/schedule.py) */
#define QB_K_NONE 0
#define QB_K_REG 1    /* pos = index into the pass's reg_bits            */
#define QB_K_THREAD 2 /* pos = tile-local bit held in the thread index   */
#define QB_K_EXT 3    /* pos = global qubit outside the tile             */

#define QB_PASS_WARP_LOCAL 1

#define QB_OP_DENSE 0 /* e^{i gamma} U(theta,phi,lam) on target [, control]            */
#define QB_OP_DIAG 1  /* diag(e^{i gamma}, e^{i(gamma+lam)}) on target [, control]     */

/* --- sweep program records (flat arrays produced by the host-side planner) ------------------------- */
typedef struct qb_sweep {
    int32_t tile_qubits[16]; /* first tile_bits entries used, ascending; tile-local bit i <-> this qubit */
    int32_t pass_begin, pass_end;
    int32_t op_begin, op_end; /* pass-op range of the whole sweep = [passes[pass_begin].op_begin, passes[pass_end-1].op_end) */
} qb_sweep;

typedef struct qb_pass {
    int32_t reg_bits[7]; /* tile-local bit positions held in registers (first reg_bits entries used) */
    int32_t flags;       /* bit 0 (QB_PASS_WARP_LOCAL): the next pass keeps the same tile bits on the warp-index bits, so the
                            shared-memory exchange after this pass needs __syncwarp only */
    int32_t op_begin, op_end;
    uint8_t thread_bits[12]; /* tile-local bit carried by thread-index bit i (the tile_bits - reg_bits others) */
} qb_pass;

typedef struct qb_pass_op {
    int32_t op_index; /* index into the circuit's op table (selects the bound 2x2 matrix) */
    uint8_t kind;     /* QB_OP_*  */
    uint8_t tgt_kind, tgt_pos;
    uint8_t ctrl_kind, ctrl_pos;
    /* pre-decoded operands (derived from the fields above; checked by qb_plan_create; the kernel builds its own dispatch word
     * from the descriptive fields when it stages a sweep, these stay for host-side tools):
     *   variant     dense: 6 * target_reg_bit + (control_reg_bit + 1)           (0..29)
     *               diag : 32 = target outside registers, 33 + b = target register bit b, both without a
     *                      register control; 40 = generic (register-controlled) diagonal
     *   ctrl_qubit  global qubit index of a QB_K_THREAD / QB_K_EXT control, 0xFF otherwise
     *   tgt_qubit   global qubit index of a QB_K_THREAD / QB_K_EXT diagonal target, 0xFF otherwise */
    uint8_t variant, ctrl_qubit, tgt_qubit;
} qb_pass_op;

/* angle sources of one op: value_j = cnst[j] + coeff[j] * params[slot[j]] + coeff2[j] * params[slot2[j]]  (slot < 0: no such
 * term); j = 0..3 -> gamma, theta, phi, lam.  This is where the flat parameter vector of
 * circuit_evaluation.py:205-207 is bound ([upstream] EstimatorPub.coerce order = sorted parameter names).  The second term
 * carries the deferred trailing phase of the previous gate on the same qubit (queasars_b200/gate_list.py: defer_phases). */
typedef struct qb_op_angles {
    int32_t slot[4];
    int32_t slot2[4];
    double coeff[4];
    double coeff2[4];
    double cnst[4];
    int32_t kind;
    int32_t pad;
} qb_op_angles;

typedef struct qb_context qb_context;

/* --- context ---------------------------------------------------------------------------------------- */
/* One engine per (process, device).  `stream` = an existing cudaStream_t to launch on (e.g. torch's), or
 * NULL to let the context create its own non-blocking stream. */
int qb_device_count(int* out); /* CUDA devices visible to the process (device sets of the multi-GPU primitives) */
int qb_context_create(int device, void* stream, qb_context** out);
int qb_context_destroy(qb_context* ctx);
const char* qb_last_error(void);
/* cudaStream_t the context launches on (for CUDA-event timing by the caller). */
void* qb_context_stream(qb_context* ctx);
/* Number of kernels this context has launched so far (bench.py's gpu_launches). */
int64_t qb_context_launch_count(qb_context* ctx);
/* Streaming multiprocessors of the context's device (chunk sizing of the pipelined submission). */
int qb_context_sm_count(qb_context* ctx);
/* Upper bound for statevector workspace (bytes); 0 = 80 % of the device memory free at creation. */
int qb_context_set_workspace_limit(qb_context* ctx, uint64_t bytes);
/* The limit in effect (bytes): a statevector larger than this does not fit one device and has to be sharded. */
uint64_t qb_context_workspace(qb_context* ctx);
/* Amplitude-index width of the sweep kernels: 32 = automatic (32-bit indices up to 31 local qubits, 64-bit above: the shards of
 * BASELINE config C5), 64 = always the 64-bit-index kernels, so that the kernels a 35-qubit sharded state runs can be checked
 * against the oracle at sizes the oracle finishes in seconds. */
int qb_context_set_index_width(qb_context* ctx, int bits);
int qb_context_synchronize(qb_context* ctx);

/* --- plans: a parsed + scheduled circuit --------------------------------------------------------------
 * Replaces TranspilingEstimatorV2/SamplerV2.run's per-call PassManager.run
 * (circuit_evaluation/transpiling_primitives.py:47, 73-80) and the upstream per-call circuit binding:
 * the circuit is compiled once, parameters are bound on the device at evaluation time. */
int qb_plan_create(qb_context* ctx, int n_qubits, int dtype, int tile_bits, int reg_bits, int n_params,
                   int n_ops, const qb_op_angles* ops,
                   int n_sweeps, const qb_sweep* sweeps,
                   int n_passes, const qb_pass* passes,
                   int n_pass_ops, const qb_pass_op* pass_ops,
                   const int32_t* init_ops /* max(n_qubits, tile_bits) entries or NULL: product-state start, see below */,
                   int64_t* plan_id);
/* init_ops[q] >= 0: qubit q starts in the first column of op init_ops[q]'s bound matrix instead of |0> (the planner
 * peels uncontrolled first gates off the circuit and drops controlled gates whose control is still |0>); the first
 * sweep then synthesises the product state prod_q v_q[bit_q(k)] instead of |0...0>.  Such ops must not appear in
 * any pass. */
int qb_plan_destroy(qb_context* ctx, int64_t plan_id);
/* Prefix-state reuse (SURVEY.md section 8f-1; the optimizer loop of evqe/evolutionary_algorithm/mutation.py:57-81 re-evaluates
 * ONE circuit whose leading layers are bound numerically and only one layer's parameters change): `plan_id` (compiled
 * for application to an existing state, no parameters in the prefix) starts from the state produced by the
 * parameter-free plan `prefix_plan_id` instead of |0...0>.  The prefix state is computed once, on first use, and kept on
 * the device (16 B * 2^n) until the plan is destroyed. */
int qb_plan_set_prefix(qb_context* ctx, int64_t plan_id, int64_t prefix_plan_id);

/* --- Hamiltonians ---------------------------------------------------------------------------------------
 * H = sum_t (coeff_re[t] + i coeff_im[t]) * P_t with P_t = i^{popcount(x&z)} X^{x_mask} Z^{z_mask}
 * (the SparsePauliOp handed to OperatorCircuitEvaluator, circuit_evaluation.py:181-198).
 * build_table != 0 precomputes the diagonal part E(k) = sum_t c_t (-1)^{popcount(k & z_t)} as an fp64 table
 * of 2^n entries ([upstream] _evaluate_sparsepauli / sampled_expectation_value semantics). */
int qb_hamiltonian_create(qb_context* ctx, int n_qubits, int n_terms,
                          const uint64_t* x_masks, const uint64_t* z_masks,
                          const double* coeff_re, const double* coeff_im,
                          int build_table, int64_t* ham_id);
int qb_hamiltonian_destroy(qb_context* ctx, int64_t ham_id);
/* E(k) for a list of basis states (sampler routes: expectation_calculation.py:60-66). */
int qb_hamiltonian_diag_energies(qb_context* ctx, int64_t ham_id, int64_t n_states,
                                 const uint64_t* states, double* out_energies);

/* --- batched evaluation ---------------------------------------------------------------------------------
 * One call = the batched submission of a generation's circuits: entry i evaluates plan_ids[i] with the
 * parameter vector params[param_offsets[i] .. param_offsets[i+1]).
 *
 * qb_evaluate_expectation  <->  OperatorCircuitEvaluator.evaluate_circuits (circuit_evaluation.py:200-215)
 *   + [upstream] StatevectorEstimator._run_pub with precision = 0:  out[i] = Re <psi_i|H|psi_i>.
 * qb_sample  <->  measure_quasi_distributions (circuit_evaluation.py:29-59) + [upstream]
 *   StatevectorSampler._run_pub / Generator.choice: out_indices[i*shots + s] =
 *   searchsorted(cumsum(|psi_i|^2)/sum, uniforms[i*shots + s], side='right').
 * qb_statevector: amplitudes of one bound circuit as complex128 (testing / debugging). */
int qb_evaluate_expectation(qb_context* ctx, int batch, const int64_t* plan_ids,
                            const double* params, const int64_t* param_offsets,
                            int64_t ham_id, double* out_values);
int qb_sample(qb_context* ctx, int batch, const int64_t* plan_ids,
              const double* params, const int64_t* param_offsets,
              int shots, const double* uniforms, int64_t* out_indices);
int qb_statevector(qb_context* ctx, int64_t plan_id, const double* params, int n_params,
                   double* out_re_im /* 2 * 2^n doubles */);

/* qb_evaluate_cvar  <->  OperatorSamplerCircuitEvaluator / BitstringCircuitEvaluator with CVaR(alpha) on the exact
 * distribution instead of shots: out[i] = expectation.lower_tail_expectation_arrays(|psi_i|^2, E, alpha) over all 2^n basis
 * states, E(k) = sum_t c_t (-1)^{popcount(k & z_t)} -- the lower alpha tail of |psi_i|^2 in stable ascending (E(k), k) order,
 * greedy fill stopped once the mass is numpy.isclose to alpha, divided by alpha.  With alpha isclose to 1 the fill runs in basis
 * order (no sort), as in that function.  The Hamiltonian must be diagonal (QB_ERR_INVALID otherwise, and for alpha outside
 * (0, 1], when a plan's width or dtype differs from the first plan's or the Hamiltonian's, and for alpha < 1 on more than 32
 * qubits: the sorted order stores 32-bit basis indices).  Its data is built on first use
 * and kept until the Hamiltonian is destroyed: E in basis order (8 B per amplitude), and for alpha < 1 the sorted order and E
 * sorted (12 B more); QB_ERR_MEMORY when it does not fit the workspace.  Deterministic: bit-identical across runs and
 * independent of the other entries of the batch. */
int qb_evaluate_cvar(qb_context* ctx, int batch, const int64_t* plan_ids, const double* params,
                     const int64_t* param_offsets, int64_t ham_id, double alpha, double* out_values);

/* --- observable sets ------------------------------------------------------------------------------------
 * Several observables H_j = sum_t c_{j,t} P_t evaluated on one simulated state (EstimatorV2 pubs with an array of observables).
 * Observable j owns the terms term_offsets[j] .. term_offsets[j+1]-1 of the mask / coefficient arrays (term_offsets[0] == 0).
 * qb_observables_create builds the union of the distinct (x, z) strings of all observables, the rows that combine them
 * (duplicate strings of one observable summed, ascending union order), and plans the strings' x-mask groups into tile sweeps as
 * qb_hamiltonian_create does.  coeff_im may be null: every P_t is Hermitian, so only Re(c_{j,t}) enters Re<psi|H_j|psi>.
 * QB_ERR_INVALID for n_obs < 1, decreasing offsets or a string outside the register.
 * qb_evaluate_observables: out_values[i * n_obs + j] = Re <psi_i|H_j|psi_i> = sum_t Re(c_{j,t}) <psi_i|P_t|psi_i> (row-major,
 * batch x n_obs), the semantics of qb_evaluate_expectation per observable.  Every distinct string is reduced once per state:
 * one read of the state per tile sweep of x-mask groups (plus two reads per 8 strings of a group wider than a tile), each
 * string into its own per-CTA partials, summed in a fixed order -- no atomics, bit-identical across runs, batch compositions
 * and workspace limits.  A list that does not fit the workspace is evaluated in chunks; QB_ERR_MEMORY (with byte counts) only
 * when one statevector and its scratch do not fit.  QB_ERR_INVALID when a plan's width differs from the set's or a plan's
 * width or dtype from the first plan's. */
int qb_observables_create(qb_context* ctx, int n_qubits, int n_obs, const int64_t* term_offsets /* n_obs + 1 */,
                          const uint64_t* x_masks, const uint64_t* z_masks, const double* coeff_re, const double* coeff_im,
                          int64_t* obs_id);
int qb_observables_destroy(qb_context* ctx, int64_t obs_id);
int qb_evaluate_observables(qb_context* ctx, int batch, const int64_t* plan_ids, const double* params,
                            const int64_t* param_offsets, int64_t obs_id, double* out_values /* batch * n_obs, row-major */);

/* One evaluate_circuits() list split over several GPUs of one process (the device sets of queasars_b200/primitives.py: the
 * reference wraps ONE primitive in a ThreadPoolExecutor, evqe.py:232-236): entry i of every array belongs to context ctxs[i] and
 * has the meaning of the corresponding qb_evaluate_expectation argument.  Every context evaluates its share on its own host
 * thread (created on first use, owned by the context), so the devices are fed concurrently and outside a Python caller's
 * interpreter lock; returns when all shares are done.  A context may appear once per call; concurrent calls on disjoint
 * context sets are fine, calls that share a context are serialised by the caller. */
int qb_evaluate_expectation_multi(int n_ctx, qb_context* const* ctxs, const int* batches, const int64_t* const* plan_ids,
                                  const double* const* params, const int64_t* const* param_offsets, const int64_t* ham_ids,
                                  double* const* out_values);

/* Pipelined form of qb_evaluate_expectation for one evaluate_circuits() list handed over in chunks: _submit queues a chunk
 * (upload, kernels, download into a pinned buffer) and returns without waiting, so the caller can prepare the next chunk's
 * parameter values (in QUEASARS: Python lists of floats, circuit_evaluation.py:205-207) while the GPU works; _collect waits
 * for everything queued on this context since the last collect and returns the `total` values in submission order.  All
 * chunks of one list must be submitted and collected by one thread without other submissions in between. */
int qb_evaluate_expectation_submit(qb_context* ctx, int batch, const int64_t* plan_ids,
                                   const double* params, const int64_t* param_offsets, int64_t ham_id);
int qb_evaluate_expectation_collect(qb_context* ctx, int total, double* out_values);

/* --- resident batches (benchmarks, optimizer inner loops) ---------------------------------------------
 * Same work as qb_evaluate_expectation split into its host<->device and device-only parts so the
 * device-resident throughput can be timed separately from the end-to-end call. */
int qb_batch_create(qb_context* ctx, int batch, const int64_t* plan_ids, int64_t ham_id, int64_t* batch_id);
int qb_batch_set_params(qb_context* ctx, int64_t batch_id, const double* params, const int64_t* param_offsets);
int qb_batch_run(qb_context* ctx, int64_t batch_id);   /* asynchronous on the context's stream */
int qb_batch_read(qb_context* ctx, int64_t batch_id, double* out_values); /* synchronises */
int qb_batch_destroy(qb_context* ctx, int64_t batch_id);
/* sweep launches / algorithmic bytes of one qb_batch_run (for roofline accounting) */
int qb_batch_stats(qb_context* ctx, int64_t batch_id, int64_t* n_sweep_launches, int64_t* n_state_sweeps,
                   int64_t* sweep_bytes, int64_t* n_kernel_launches);

/* Like qb_batch_run, with a CUDA event pair around every sweep-kernel launch (same stream): fills the
 * device time of each sweep launch in milliseconds and the number of statevectors it swept; synchronises.
 * Used by bench.py to compute the live roofline of the dominant kernel. */
int qb_batch_run_timed(qb_context* ctx, int64_t batch_id, int max_launches, float* sweep_ms, int32_t* sweep_states,
                       int* n_launches);

/* --- device-pointer entry points (parity tests, sharded multi-GPU path) -------------------------------
 * Operate on a caller-owned device statevector of 2^n_local amplitudes.  `index_offset` is OR-ed into the
 * amplitude index seen by QB_K_EXT operands and by the diagonal table lookup, so a rank holding the shard
 * with global-qubit bits `rank << n_local` evaluates controls on global qubits correctly.  A plan whose width is below
 * its sweep tile (2^tile_bits amplitudes) is refused by qb_apply_plan_device with QB_ERR_INVALID: its sweeps would cover
 * more than the caller's buffer. */
int qb_apply_plan_device(qb_context* ctx, int64_t plan_id, const double* params_host, int n_params,
                         void* d_state, int init_zero_state, uint64_t index_offset);
int qb_expectation_device(qb_context* ctx, int64_t ham_id, int dtype, int n_local, const void* d_state,
                          uint64_t index_offset, double* out_value);
/* qb_sample on a caller-owned (possibly un-normalised: a shard) device state of 2^n_local amplitudes:
 * out_indices[s] = searchsorted(cumsum(|psi|^2) / sum, uniforms[s], side='right').  The sharded sampler
 * (queasars_b200/sharded.py) first picks the shard of every shot from the all-gathered shard masses and hands each
 * rank its shots with re-scaled uniforms ([upstream] StatevectorSampler / Generator.choice semantics per shard). */
int qb_sample_device(qb_context* ctx, int dtype, int n_local, const void* d_state, int shots,
                     const double* uniforms, int64_t* out_indices);
/* One radix-digit pass of the exact CVaR of a sharded state (sort-free weighted selection, queasars_b200/sharded.py) on a
 * caller-owned shard of 2^n_local amplitudes whose physical indices are `index_offset | k`.  Entries are keyed by
 * (energy_key(E(k)), logical k) with E(k) of the diagonal Hamiltonian `ham_id` (built with physical z masks), summed like
 * qb_hamiltonian_diag_energies, and energy_key the order-preserving 64-bit image of the double (-0.0 keyed as +0.0).  Only
 * entries matching the prefix are counted: energy key >> e_free == e_prefix (e_free = 64: no energy constraint) and
 * (physical index & idx_mask) == idx_value.  The digit is bits [e_free - digit_bits, e_free) of the energy key (digit_kind 0) or
 * the physical index bits digit_positions[0..digit_bits) (digit_kind 1; the logical index bits of the digit, lowest first),
 * digit_bits <= 8.  Per bucket b of the digit: out_sums[b] = mass, out_sums[256 + b] = sum p * E (fixed summation order: the
 * same on every call), out_ints[b] = count, [256 + b] / [512 + b] = min / max energy key, [768 + b] = least physical index.
 * cache_mode 1 also writes (p, E) of every entry as two doubles into d_cache (2^n_local * 16 B, e.g. the idle spare shard
 * buffer); cache_mode 2 reads them from there and does not touch d_state.  QB_ERR_INVALID for a non-diagonal Hamiltonian, a
 * bad bit map or a bad digit.  Synchronous. */
int qb_cvar_select_device(qb_context* ctx, int64_t ham_id, int dtype, int n_local, const void* d_state, uint64_t index_offset,
                          void* d_cache, int cache_mode, uint64_t e_prefix, int e_free, int digit_kind, int digit_bits,
                          const int32_t* digit_positions, uint64_t idx_mask, uint64_t idx_value, double* out_sums,
                          uint64_t* out_ints);

/* Global <-> local qubit swap of a state sharded over `world` = 2^n_global GPUs of one node (BASELINE config C5), fused with its
 * all-to-all: the calling rank streams its shard `d_state` once and stores every amplitude directly into the rank that owns it
 * afterwards -- peer_dst[d] is rank d's destination buffer mapped into this process (peer memory over NVLink 5 / NVSwitch, e.g.
 * torch symmetric memory; peer_dst[rank] = the caller's own spare buffer) -- at its final index: amplitude i with local bits
 * local_positions[j] = d_j goes to rank d, index i with those bits replaced by the bits of `rank`.  Replaces pack +
 * ncclAllToAll + unpack.  Asynchronous on the context's stream; the caller synchronises and runs a cross-rank barrier before any
 * rank touches its destination buffer. */
int qb_swap_global_p2p(qb_context* ctx, int dtype, int n_local, const void* d_state, void* const* peer_dst, int world, int rank,
                       int n_global, const int32_t* local_positions);

/* --- device memory and peer mapping for sharded states ----------------------------------------------------
 * The shard buffers of a state sharded over several GPUs are plain cudaMalloc allocations owned by the engine of their device.
 * Single process, several GPUs (the configuration behind evaluate_circuits): qb_enable_peer_access lets the swap kernel of
 * one device store into the buffers of the others through their ordinary (unified) addresses.  One process per GPU: the owner
 * exports a CUDA IPC handle (64 opaque bytes, sent to the peers by any means, e.g. a torch.distributed all_gather) and each
 * peer maps the buffer with qb_ipc_open; the mapped address is what qb_swap_global_p2p takes in peer_dst[]. */
int qb_device_alloc(qb_context* ctx, uint64_t bytes, void** out_ptr);
int qb_device_free(qb_context* ctx, void* ptr);
/* copy `bytes` from device address `src` (+ byte offset) to host memory; synchronises (tests, gathers of small states) */
int qb_device_read(qb_context* ctx, const void* src, uint64_t offset, uint64_t bytes, void* host_out);
int qb_enable_peer_access(qb_context* ctx, int peer_device); /* QB_OK also when access was already enabled or peer == own device */
int qb_ipc_export(qb_context* ctx, void* ptr, unsigned char handle_out[64]);
int qb_ipc_open(qb_context* ctx, const unsigned char handle[64], void** out_ptr);
int qb_ipc_close(qb_context* ctx, void* mapped_ptr);

/* layout self-check for language bindings: sizeof() of the four records above */
void qb_record_sizes(int32_t out[4]);

#ifdef __cplusplus
}
#endif
#endif /* QUEASARS_B200_H */
