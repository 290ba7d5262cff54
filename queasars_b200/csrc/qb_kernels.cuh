// Hand-written sm_100a kernels of the EVQE circuit-evaluation hot path.
//
//   sweep_kernel        K1/K2  fused multi-gate application: one read + one write of the state per sweep,
//                              gates applied in registers (2^4 amplitudes / thread), passes exchanged through
//                              XOR-swizzled shared memory; optional fused diagonal-expectation epilogue (K3)
//   bind_kernel                flat parameter vector -> 2x2 matrices, on the device
//   diag_table_kernel   K3     E(k) = sum_t c_t (-1)^{popcount(k & z_t)}
//   expect_table_kernel K3     sum_k |psi_k|^2 E(k)
//   expect_group_kernel K4     Re sum_k psi_k conj(psi_{k^x}) W_x(k) for one x-mask group of a Pauli sum
//   expect_tile_kernel  K4     the same for all groups that fit one 2^11 tile: one read of the state per tile sweep
//   chunk_prob_kernel / scan_chunks_kernel / sample_kernel   K5  prefix-sum CDF sampling
//   cvar_chunk_kernel / scan_chunks_kernel / cvar_finish_kernel  K6  exact CVaR(alpha) of a diagonal Hamiltonian (sorted lower tail)
//   cvar_select_kernel / cvar_select_reduce_kernel  K8  one radix-digit pass of the exact CVaR of a sharded state (weighted select)
//   top_select_kernel / top_collect_kernel  K9  most probable basis states: counts-only radix select of (~bits(p), logical k), ordered collect
//   swap_p2p_kernel            global <-> local qubit swap of a sharded state fused with its all-to-all (peer-memory stores)
//   swap_inplace_p2p_kernel    the same exchange in place, one buffer per rank (pairs swapped by peer loads + stores)
//
// What the arithmetic follows ([upstream] = un-vendored qiskit 2.4.2, see oracle/qiskit_semantics.py):
//   gate matrices   UGate / CU3Gate as emitted by evqe/quantum_circuit/quantum_gate.py:96-102, 157-165
//   expectation     circuit_evaluation/circuit_evaluation.py:200-215 -> [upstream] Statevector.expectation_value
//   sampling        circuit_evaluation/circuit_evaluation.py:29-59 -> [upstream] Statevector.sample_memory
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "queasars_b200.h"

namespace qb {

// Build-time experiment switches (defaults are the measured best; tools/build_variants.py builds A/B libraries):
//   QB_SWEEP_CTAS   resident sweep CTAs per SM with 2^11-amplitude tiles (4 -> 128 registers per thread, 3 -> 168)
//   QB_DENSE_GROUP  amplitude pairs of a dense gate advanced together, stage by stage (independent FP64 chains per warp = 4 x this)
#ifndef QB_SWEEP_CTAS
#define QB_SWEEP_CTAS 4
#endif
#ifndef QB_DENSE_GROUP
#define QB_DENSE_GROUP 1
#endif
// Run-time launch flags of sweep_kernel
//   QB_SWEEP_L2_PREFETCH  while a CTA works on tile i it asks the L2 to fetch tile i + 1 from HBM (prefetch.global.L2, one 256-byte
//                         run per thread), so the next tile's register loads hit L2 instead of paying the HBM latency.
//                         Measured (per-lane line prefetches): +3..6 % on the read+write sweeps of 26-30-qubit states, neutral on
//                         batches of 20-qubit states; on by default (QB_L2_PREFETCH=0 switches it off).  The bulk form
//                         (cp.async.bulk.prefetch.L2 -> UBLKPF) takes a warp-uniform address and was issued lane by lane: -2 %.
constexpr int QB_SWEEP_L2_PREFETCH = 1;

constexpr int kMaxSweepOps = 96;
constexpr int kMaxSweepPasses = 16;


template <typename T> struct Cx;
template <> struct Cx<double> { using type = double2; };
template <> struct Cx<float> { using type = float2; };

// One circuit evaluation inside a batched launch.
struct BatchEntry {
    const qb_sweep* sweeps;
    const qb_pass* passes;
    const qb_pass_op* pass_ops;
    const qb_op_angles* angles;
    const int32_t* init_ops;   // device, n_eff entries (product-state start) or nullptr
    const double* params;      // device, n_params
    double* matrices;          // device: 8 doubles per op (by op index), 8 per pass-op (pass order), 4 per qubit (initial state)
    void* state;               // device, 2^n_eff amplitudes
    const void* src_state;     // optional: the first sweep reads this (cached prefix state) instead of `state`
    const double* diag_table;  // device, 2^n_eff doubles, or nullptr
    double* partials;          // device, one double per tile (fused expectation epilogue)
    int32_t n_sweeps, n_ops, n_params, init_zero;
    int32_t n_pass_ops, n_init;  // n_init = number of init_ops entries (= padded qubit count)
    uint64_t index_offset;
};

// XOR-fold of the tile-local index in groups of three bits: linear over GF(2), so
// swz(a | b) == swz(a) ^ swz(b) for disjoint a, b.  Keeps 128-bit accesses of a quarter warp on eight
// different 16-byte bank groups for every pass layout the planner emits (schedule.py:_thread_bit_order).
__device__ __forceinline__ uint32_t swz(uint32_t e) { return e ^ (((e >> 3) ^ (e >> 6) ^ (e >> 9)) & 7u); }

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Deterministic block sum (fixed tree): result valid in thread 0.
__device__ __forceinline__ double block_sum(double v, double* s_red) {
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) s_red[warp] = v;
    __syncthreads();
    double total = 0.0;
    if (threadIdx.x == 0) {
        const int nw = (blockDim.x + 31) >> 5;
        for (int w = 0; w < nw; ++w) total += s_red[w];
    }
    __syncthreads();
    return total;
}

// Explicit global-space 128-bit / 64-bit accesses (the state pointer comes out of a struct in memory, which
// the compiler would otherwise treat as a generic address).  The loads are `asm volatile`: a plain asm is "pure" to the
// compiler, which may then hoist it above the condition that guards it (seen: the diagonal-table load speculated with a
// null table pointer).
// Programmatic dependent launch (sm_90+): a kernel launched with the programmatic-stream-serialization attribute may start while
// its predecessor in the stream still runs; everything it reads that the predecessor (or anything before it) wrote has to come
// after pdl_wait(), which returns once the predecessor grids have completed and their writes are visible.  Both are no-ops in
// a kernel launched the ordinary way.  Data read behind pdl_wait() is loaded with .cg (L2 only): the kernel's lifetime
// overlaps the writes, so neither the non-coherent path nor a line left in L1 by an earlier grid may serve it.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ double ld_cg(const double* p) {
    double r;
    asm volatile("ld.global.cg.f64 %0, [%1];" : "=d"(r) : "l"(p));
    return r;
}

#ifndef QB_PLAIN_FAST
#define QB_PLAIN_FAST 1
#endif
#ifndef QB_TABLE_LD
#define QB_TABLE_LD "ld.global.nc.f64"
#endif
#ifndef QB_STATE_LD
#define QB_STATE_LD "ld.global.cg"
#endif
__device__ __forceinline__ double2 ld_state(const double2* p) {
    double2 r;
    asm volatile(QB_STATE_LD ".v2.f64 {%0, %1}, [%2];" : "=d"(r.x), "=d"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ float2 ld_state(const float2* p) {
    float2 r;
    asm volatile(QB_STATE_LD ".v2.f32 {%0, %1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ void st_state(double2* p, double2 v) {
    asm volatile("st.global.v2.f64 [%0], {%1, %2};" ::"l"(p), "d"(v.x), "d"(v.y) : "memory");
}
__device__ __forceinline__ void st_state(float2* p, float2 v) {
    asm volatile("st.global.v2.f32 [%0], {%1, %2};" ::"l"(p), "f"(v.x), "f"(v.y) : "memory");
}
__device__ __forceinline__ double ld_table(const double* p) {
    double r;
    asm volatile(QB_TABLE_LD " %0, [%1];" : "=d"(r) : "l"(p));
    return r;
}

// 2x2 complex matrix on register bit B of the 16 register-resident amplitudes.  CB >= 0: controlled by register
// bit CB (only the 4 pairs with that bit set are touched); CB < 0: all 8 pairs.  Everything is resolved at compile
// time so the 8 (4) pair updates are straight-line code the scheduler can interleave (no per-pair predicates).
// REAL00: the matrix's top-left entry is real (every gate without a global phase, e^{i gamma} = 1: all of EVQE's u / cu3) -- two of
// the sixteen multiply-adds per pair vanish.  The flag is a property of the plan (gamma identically 0), so it is part of the
// dispatch word; skipping the two FMAs is bit-identical to executing them with m00.y = +0.
// REAL10: the bottom-left entry is real as well (phi == 0: the R_Y(theta) * D(lam) form every uncontrolled gate has after the
// front end's phase deferral, gate_list.py: defer_phases) -- two more multiply-adds vanish, 12 per pair.
template <typename T, int R, int B, int CB, bool REAL00 = false, bool REAL10 = false>
__device__ __forceinline__ void apply_dense(typename Cx<T>::type (&a)[1 << R], const typename Cx<T>::type m00, const typename Cx<T>::type m01,
                                            const typename Cx<T>::type m10, const typename Cx<T>::type m11) {
    constexpr int kNReg = 1 << R;
    constexpr int kPairs = (CB >= 0) ? kNReg / 4 : kNReg / 2;
    constexpr int G = (QB_DENSE_GROUP < kPairs) ? QB_DENSE_GROUP : kPairs;
    using C = typename Cx<T>::type;
#if QB_DENSE_GROUP == 1
    // Term order chosen so that the last FMA of each output reads exactly the register it overwrites: the update is in place
    // with four temporaries and no register moves at loop / switch merge points.
#pragma unroll
    for (int j = 0; j < kNReg; ++j) {
        if (j & (1 << B)) continue;
        if (CB >= 0 && !(j & (1 << (CB >= 0 ? CB : 0)))) continue;
        const C x = a[j], y = a[j | (1 << B)];
        T t0 = m01.x * y.x;
        T t1 = m01.x * y.y;
        T t2 = m10.x * x.x;
        T t3 = m10.x * x.y;
        t0 = fma(-m01.y, y.y, t0);
        t1 = fma(m01.y, y.x, t1);
        if (!REAL10) {
            t2 = fma(-m10.y, x.y, t2);
            t3 = fma(m10.y, x.x, t3);
        }
        if (!REAL00) {
            t0 = fma(-m00.y, x.y, t0);
            t1 = fma(m00.y, x.x, t1);
        }
        t2 = fma(-m11.y, y.y, t2);
        t3 = fma(m11.y, y.x, t3);
        a[j].x = fma(m00.x, x.x, t0);
        a[j].y = fma(m00.x, x.y, t1);
        a[j | (1 << B)].x = fma(m11.x, y.x, t2);
        a[j | (1 << B)].y = fma(m11.x, y.y, t3);
    }
    return;
#endif
    // compile-time list of the pair bases this gate touches (register index with bit B clear, and bit CB set when controlled)
    int base[kPairs];
    {
        int n = 0;
#pragma unroll
        for (int j = 0; j < kNReg; ++j) {
            if (j & (1 << B)) continue;
            if (CB >= 0 && !(j & (1 << (CB >= 0 ? CB : 0)))) continue;
            base[n++] = j;
        }
    }
    // Term order chosen so that the last FMA of each output reads exactly the register it overwrites: the update is in place
    // with four temporaries per pair and no register moves at loop / switch merge points.  G pairs advance together, one
    // multiply-add stage at a time, so a warp carries 4 * G independent FP64 chains.
#pragma unroll
    for (int g0 = 0; g0 < kPairs; g0 += G) {
        T t0[G], t1[G], t2[G], t3[G];
#pragma unroll
        for (int g = 0; g < G; ++g) {
            const C x = a[base[g0 + g]], y = a[base[g0 + g] | (1 << B)];
            t0[g] = m01.x * y.x;
            t1[g] = m01.x * y.y;
            t2[g] = m10.x * x.x;
            t3[g] = m10.x * x.y;
        }
#pragma unroll
        for (int g = 0; g < G; ++g) {
            const C y = a[base[g0 + g] | (1 << B)];
            t0[g] = fma(-m01.y, y.y, t0[g]);
            t1[g] = fma(m01.y, y.x, t1[g]);
        }
        if (!REAL10) {
#pragma unroll
            for (int g = 0; g < G; ++g) {
                const C x = a[base[g0 + g]];
                t2[g] = fma(-m10.y, x.y, t2[g]);
                t3[g] = fma(m10.y, x.x, t3[g]);
            }
        }
        if (!REAL00) {
#pragma unroll
            for (int g = 0; g < G; ++g) {
                const C x = a[base[g0 + g]];
                t0[g] = fma(-m00.y, x.y, t0[g]);
                t1[g] = fma(m00.y, x.x, t1[g]);
            }
        }
#pragma unroll
        for (int g = 0; g < G; ++g) {
            const C y = a[base[g0 + g] | (1 << B)];
            t2[g] = fma(-m11.y, y.y, t2[g]);
            t3[g] = fma(m11.y, y.x, t3[g]);
        }
#pragma unroll
        for (int g = 0; g < G; ++g) {
            const int j = base[g0 + g];
            const C x = a[j], y = a[j | (1 << B)];
            a[j].x = fma(m00.x, x.x, t0[g]);
            a[j].y = fma(m00.x, x.y, t1[g]);
            a[j | (1 << B)].x = fma(m11.x, y.x, t2[g]);
            a[j | (1 << B)].y = fma(m11.x, y.y, t3[g]);
        }
    }
}

template <typename T>
__device__ __forceinline__ typename Cx<T>::type cmul(typename Cx<T>::type a, typename Cx<T>::type b) {
    typename Cx<T>::type r;
    r.x = a.x * b.x - a.y * b.y;
    r.y = a.x * b.y + a.y * b.x;
    return r;
}

// XOR of the per-register-bit offsets selected by the compile-time register index j (global offsets are
// disjoint bits, swizzled shared-memory offsets are not: XOR is right for both)
template <int R, typename U>
__device__ __forceinline__ U reg_offset(int j, const U (&off)[R]) {
    U r = 0;
#pragma unroll
    for (int i = 0; i < R; ++i)
        if (j & (1 << i)) r ^= off[i];
    return r;
}

// ---------------------------------------------------------------------------------------------------
// sweep kernel: grid = (tiles >> m_log2, active batch entries), block = 2^(K-R) threads, dynamic smem = sweep_smem_bytes<T, R, K>()
//
// Every CTA stages the sweep program of ITS circuit once -- pass records, matrices, one pre-decoded dispatch word per op, the
// per-pass thread -> tile-slot table -- and then walks 2^m_log2 consecutive tiles with it, so the dependent-load prologue and
// all per-pass index arithmetic are paid once per CTA instead of once per tile.  Per tile only the operands that live outside
// the tile (controls / diagonal targets on non-tile qubits) are re-resolved, by one thread per op, into a double-buffered word
// list; the single CTA barrier per tile that publishes it sits behind the issue of the tile's HBM loads.
// ---------------------------------------------------------------------------------------------------
constexpr int kWordStride = kMaxSweepOps + 1;
constexpr int kMaxInitQubits = 64;

// dispatch word: variant | cpos << 6 | dpos << 11 | dflag << 16 | cb << 17 | tb << 20 | treg << 23
//   variant bit 5 (dense ops): the matrix's top-left entry is real (gamma == 0) -> 14 instead of 16 multiply-adds per pair
//   variant 48 + b (uncontrolled dense on register bit b): the whole first column is real (gamma == phi == 0) -> 12; with bit 31
//         (QB_PLAIN_FAST) the op loop runs it in tangent form instead -> 8 (apply_tangent)
//   cpos  tile-local position of a thread-bit control; 31 = none (bit 31 of the test word is always set), 30 = an external
//         control that is 0 for this tile (bit 30 is never set)
//   dpos  tile-local position of a thread-bit diagonal target; 31 = use dflag (external target, resolved per tile)
//   cb / tb / treg  register-bit control / register-bit target of the generic controlled diagonal
template <int R> __host__ __device__ constexpr int v_dense(int B) { return B; }
template <int R> __host__ __device__ constexpr int v_ctrl(int B, int CB) { return R + B * (R - 1) + (CB < B ? CB : CB - 1); }
template <int R> __host__ __device__ constexpr int v_diag_out() { return R * R; }
template <int R> __host__ __device__ constexpr int v_diag_reg(int b) { return R * R + 1 + b; }
template <int R> __host__ __device__ constexpr int v_diag_gen() { return R * R + 1 + R; }

template <typename T, int R, int K>
constexpr size_t sweep_smem_bytes() {
    return sizeof(typename Cx<T>::type) * (size_t(1) << K) + sizeof(T) * 8 * kMaxSweepOps + sizeof(typename Cx<T>::type) * 2 * kMaxInitQubits +
           sizeof(uint32_t) * kMaxSweepPasses * 8 + sizeof(uint32_t) * 4 * kWordStride + sizeof(qb_pass) * kMaxSweepPasses +
           sizeof(uint16_t) * kMaxSweepPasses * (size_t(1) << (K - R));
}

// apply_dense for a (B, CB) pair that may not exist for this R (keeps the case lists below uniform)
template <typename T, int R, int B, int CB, bool REAL00, bool REAL10 = false>
__device__ __forceinline__ void dense_if(typename Cx<T>::type (&a)[1 << R], const typename Cx<T>::type* __restrict__ m) {
    if constexpr (B < R && CB < R && B != CB) apply_dense<T, R, B, CB, REAL00, REAL10>(a, m[0], m[1], m[2], m[3]);
}

// uncontrolled dense gate on register bit v (< R): two predictable branches
template <typename T, int R, bool REAL00, bool REAL10 = false>
__device__ __forceinline__ void dense_by_bit(uint32_t v, typename Cx<T>::type (&a)[1 << R], const typename Cx<T>::type* __restrict__ m) {
    if (v & 2u) {
        if constexpr (R > 3) {
            if (v & 1u) dense_if<T, R, 3, -1, REAL00, REAL10>(a, m);
            else dense_if<T, R, 2, -1, REAL00, REAL10>(a, m);
        } else {
            dense_if<T, R, 2, -1, REAL00, REAL10>(a, m);
        }
    } else {
        if (v & 1u) dense_if<T, R, 1, -1, REAL00, REAL10>(a, m);
        else dense_if<T, R, 0, -1, REAL00, REAL10>(a, m);
    }
}

// Tangent form of a plain op (uncontrolled, real first column): M = [[c, -s E], [s, c E]] = c [[1, -t E], [t, E]] with t = s / c.
// The body applies the bracket -- 2 multiplies + 6 multiply-adds per pair instead of REAL10's 4 + 8 -- and the sweep multiplies
// its amplitudes by the product of the c's once before the store (sweep_kernel: stage_tangent, s_scale).  Record (staged in place
// of the op's matrix): m[0] = E, m[1].x = t.  In place with two temporaries: y is dead once w = E y is formed, x once x' is.
template <typename T, int R, int B>
__device__ __forceinline__ void apply_tangent(typename Cx<T>::type (&a)[1 << R], const typename Cx<T>::type* __restrict__ m) {
    using C = typename Cx<T>::type;
    const C e = m[0];
    const T t = m[1].x;
#pragma unroll
    for (int j = 0; j < (1 << R); ++j) {
        if (j & (1 << B)) continue;
        const C x = a[j], y = a[j | (1 << B)];
        T w0 = e.x * y.x;
        T w1 = e.x * y.y;
        w0 = fma(-e.y, y.y, w0);
        w1 = fma(e.y, y.x, w1);
        a[j | (1 << B)].x = fma(t, x.x, w0);
        a[j | (1 << B)].y = fma(t, x.y, w1);
        a[j].x = fma(-t, w0, x.x);
        a[j].y = fma(-t, w1, x.y);
    }
}

// the op loop's direct path: a tangent-form plain op on register bit v (< R), two predictable branches
template <typename T, int R>
__device__ __forceinline__ void tangent_by_bit(uint32_t v, typename Cx<T>::type (&a)[1 << R], const typename Cx<T>::type* __restrict__ m) {
    if (v & 2u) {
        if constexpr (R > 3) {
            if (v & 1u) apply_tangent<T, R, 3>(a, m);
            else apply_tangent<T, R, 2>(a, m);
        } else {
            apply_tangent<T, R, 2>(a, m);
        }
    } else {
        if (v & 1u) apply_tangent<T, R, 1>(a, m);
        else apply_tangent<T, R, 0>(a, m);
    }
}

// Amplitudes in tangent form grow by 1 / |c| per op (the norm of M / c), so the sweep keeps a plain op in that form only while
// the product of the |c|'s of its plain ops so far stays >= kTangentMinScale: amplitudes stay below 2^400 (double) / 2^40 (float),
// their squares and the pair updates finite.  The bound is a guarantee for any circuit, not a statistic of a workload.
template <typename T> struct TangentBudget;
template <> struct TangentBudget<double> { static constexpr double kMinScale = 0x1p-400; };
template <> struct TangentBudget<float> { static constexpr double kMinScale = 0x1p-40; };

// One warp, after the sweep's matrices are staged: every plain op (bit 31 of its word) within the budget gets its tangent record;
// one over the budget, or with c == 0, keeps its matrix and drops to the real-top-left body (bits 31 and 4 cleared: variant
// 48 + b -> 32 + b, which never reads m00.y).  Writes the product of the kept ops' c's (signed) to *s_scale; 1 without one.
template <typename T>
__device__ __forceinline__ void stage_tangent(typename Cx<T>::type* s_mat, uint32_t* s_word0, int n_sop, int lane, double* s_scale) {
    double carry = 1.0, scale = 1.0;
#pragma unroll 1
    for (int o0 = 0; o0 < n_sop; o0 += 32) {
        const int o = o0 + lane;
        const bool plain = o < n_sop && int32_t(s_word0[o]) < 0;
        if (!__any_sync(0xffffffffu, plain)) continue;
        typename Cx<T>::type* m = s_mat + o * 4;
        const double c = plain ? double(m[0].x) : 1.0;
        // inclusive prefix product of |c| over the sweep's plain ops, in op order (an op with c == 0 is skipped, not counted)
        double p = (c != 0.0) ? fabs(c) : 1.0;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const double q = __shfl_up_sync(0xffffffffu, p, d);
            if (lane >= d) p *= q;
        }
        p *= carry;
        carry = __shfl_sync(0xffffffffu, p, 31);
        if (plain && c != 0.0 && p >= TangentBudget<T>::kMinScale) {
            const double r = 1.0 / c;
            const double t = double(m[2].x) * r;
            typename Cx<T>::type e;
            e.x = T(double(m[3].x) * r), e.y = T(double(m[3].y) * r);
            m[0] = e;
            m[1].x = T(t);
            scale *= c;
        } else if (plain) {
            s_word0[o] &= ~(0x80000000u | 16u);
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) scale *= __shfl_xor_sync(0xffffffffu, scale, d);
    if (lane == 0) *s_scale = scale;
}

// register-controlled dense gate: c = v - R enumerates (B, CB) as B * (R - 1) + k with CB = the k-th register bit other than B;
// combinations that do not exist for this R get labels that never match
template <int R> __host__ __device__ constexpr int ctrl_label(int B, int k) { return (B < R && k < R - 1) ? B * (R - 1) + k : 100 + 4 * B + k; }

template <typename T, int R, bool REAL00>
__device__ __forceinline__ void ctrl_by_code(uint32_t c, typename Cx<T>::type (&a)[1 << R], const typename Cx<T>::type* __restrict__ m) {
    switch (c) {
#define QB_C(B, K_) case ctrl_label<R>(B, K_): dense_if<T, R, B, (K_ < B ? K_ : K_ + 1), REAL00>(a, m); break;
        QB_C(0, 0) QB_C(0, 1) QB_C(0, 2)
        QB_C(1, 0) QB_C(1, 1) QB_C(1, 2)
        QB_C(2, 0) QB_C(2, 1) QB_C(2, 2)
        QB_C(3, 0) QB_C(3, 1) QB_C(3, 2)
#undef QB_C
        default: break;
    }
}

template <typename T, int R>
__device__ __forceinline__ void apply_op(uint32_t word, uint32_t e_thr, typename Cx<T>::type (&a)[1 << R], const typename Cx<T>::type* __restrict__ m) {
    static_assert(R == 3 || R == 4, "2^3 or 2^4 amplitudes per thread");
    using C = typename Cx<T>::type;
    constexpr int kNReg = 1 << R;
    const uint32_t variant = word & 63u;
    // (matrix entries are read where a case needs them: hoisting the four 128-bit loads above the dispatch costs 16 live
    //  registers and spills -- measured -6 %)
    auto diag_select = [&]() -> C {  // factor of a diagonal whose target is not a register bit
        const uint32_t sel = ((e_thr | ((word >> 16) << 31)) >> ((word >> 11) & 31u)) & 1u;
        return sel ? m[3] : m[0];
    };
    // The common cases are reached by predictable branches instead of the jump table (+2 %), the commonest first: an
    // uncontrolled dense gate with a real first column (variants 48 + b: every `u` of an EVQE circuit after phase deferral),
    // then one with a real top-left entry only (bit 5 of the variant).
#if !QB_PLAIN_FAST
    if ((variant ^ 48u) < uint32_t(R)) {
        dense_by_bit<T, R, true, true>(variant & 3u, a, m);
        return;
    }
#endif
    if ((variant ^ 32u) < uint32_t(R)) {
        dense_by_bit<T, R, true>(variant & 3u, a, m);
        return;
    }
    if (variant & 32u) {  // controlled dense gate with a real top-left entry
        ctrl_by_code<T, R, true>((variant & 31u) - uint32_t(R), a, m);
        return;
    }
    if (variant < uint32_t(R)) {  // uncontrolled dense gate with a global phase
        dense_by_bit<T, R, false>(variant, a, m);
        return;
    }
    if (variant < uint32_t(v_diag_out<R>())) {
        ctrl_by_code<T, R, false>(variant - uint32_t(R), a, m);
        return;
    }
    if (variant == uint32_t(v_diag_out<R>())) {
        const C d = diag_select();
#pragma unroll
        for (int j = 0; j < kNReg; ++j) a[j] = cmul<T>(a[j], d);
    } else if (variant < uint32_t(v_diag_gen<R>())) {
        const uint32_t tb = 1u << (variant - uint32_t(v_diag_reg<R>(0)));
        const C d0 = m[0], d1 = m[3];
#pragma unroll
        for (int j = 0; j < kNReg; ++j) a[j] = cmul<T>(a[j], (j & tb) ? d1 : d0);
    } else if (variant == uint32_t(v_diag_gen<R>())) {  // diagonal with a register-bit control (rare: transpiled cz / cp / crz)
        const uint32_t cmask = 1u << ((word >> 17) & 7u);
        const C d0 = m[0], d1 = m[3];
        if (word & (1u << 23)) {
            const uint32_t tb = 1u << ((word >> 20) & 7u);
#pragma unroll
            for (int j = 0; j < kNReg; ++j)
                if (j & cmask) a[j] = cmul<T>(a[j], (j & tb) ? d1 : d0);
        } else {
            const C d = diag_select();
#pragma unroll
            for (int j = 0; j < kNReg; ++j)
                if (j & cmask) a[j] = cmul<T>(a[j], d);
        }
    }
}

template <typename T, int R, int K, typename Idx>
__global__ void __launch_bounds__(1 << (K - R), (K <= 11 ? QB_SWEEP_CTAS : 2))
sweep_kernel(const BatchEntry* __restrict__ entries, int sweep_idx, int n_eff, int fuse_expectation, int m_log2, int flags) {
    using C = typename Cx<T>::type;
    constexpr int kTileSize = 1 << K;
    constexpr int kThreadBits = K - R;
    constexpr int kThreads = 1 << kThreadBits;
    constexpr int kNReg = 1 << R;
    constexpr int kAmpShift = sizeof(C) == 16 ? 4 : 3;
    extern __shared__ __align__(16) unsigned char smem[];
    unsigned char* sp = smem;
    unsigned char* tile_b = sp;                                sp += sizeof(C) * kTileSize;
    C* s_mat = reinterpret_cast<C*>(sp);                       sp += sizeof(T) * 8 * kMaxSweepOps;
    C* s_init = reinterpret_cast<C*>(sp);                      sp += sizeof(C) * 2 * kMaxInitQubits;
    uint32_t* s_so = reinterpret_cast<uint32_t*>(sp);          sp += sizeof(uint32_t) * kMaxSweepPasses * 8;
    uint32_t* s_word0 = reinterpret_cast<uint32_t*>(sp);       sp += sizeof(uint32_t) * kWordStride;
    uint32_t* s_ext = reinterpret_cast<uint32_t*>(sp);         sp += sizeof(uint32_t) * kWordStride;
    uint32_t* s_word = reinterpret_cast<uint32_t*>(sp);        sp += sizeof(uint32_t) * 2 * kWordStride;
    qb_pass* s_pass = reinterpret_cast<qb_pass*>(sp);          sp += sizeof(qb_pass) * kMaxSweepPasses;
    uint16_t* s_ethr = reinterpret_cast<uint16_t*>(sp);
    __shared__ qb_sweep s_sweep;
    __shared__ uint64_t s_gi[2][8];
    __shared__ double s_red[32];
    __shared__ int s_has_ext;
    __shared__ double s_scale;  // product of the c's of the sweep's plain ops in tangent form (stage_tangent)

    pdl_launch_dependents();  // a dependent launch may start its own staging now; it waits for this grid's stores in pdl_wait()
    const BatchEntry& ge = entries[blockIdx.y];
    if (sweep_idx >= ge.n_sweeps) return;
    const int tid = threadIdx.x;

    // ================= staging (once per CTA): the sweep program first -- plan data no kernel writes =================
    if (tid < int(sizeof(qb_sweep) / 4))
        reinterpret_cast<int32_t*>(&s_sweep)[tid] = reinterpret_cast<const int32_t*>(ge.sweeps + sweep_idx)[tid];
    if (tid == 0) s_has_ext = 0;
    __syncthreads();
    const int pass_begin = s_sweep.pass_begin;
    const int n_pass = s_sweep.pass_end - pass_begin;
    const int op_begin = s_sweep.op_begin;
    const int n_sop = s_sweep.op_end - op_begin;
    const bool product_start = (sweep_idx == 0) && ge.init_zero && (ge.init_ops != nullptr);
    const bool zero_start = (sweep_idx == 0) && ge.init_zero && (ge.init_ops == nullptr);

    for (int i = tid; i < n_pass * int(sizeof(qb_pass) / 4); i += kThreads)
        reinterpret_cast<int32_t*>(s_pass)[i] = reinterpret_cast<const int32_t*>(ge.passes + pass_begin)[i];
    {
        for (int i = tid; i <= n_sop; i += kThreads) {
            uint32_t w = 0, x = 0xffffu;
            if (i < n_sop) {
                const qb_pass_op po = ge.pass_ops[op_begin + i];
                uint32_t cpos = 31, dpos = 31, cb = 0, tb = 0, treg = 0, variant, extc = 0xff, extt = 0xff;
                if (po.ctrl_kind == QB_K_THREAD) cpos = po.ctrl_pos;
                else if (po.ctrl_kind == QB_K_EXT) extc = po.ctrl_pos;
                const int rcb = (po.ctrl_kind == QB_K_REG) ? int(po.ctrl_pos) : -1;
                if (po.kind == QB_OP_DENSE) {
                    const int b = po.tgt_pos;
                    variant = rcb < 0 ? uint32_t(b) : uint32_t(R + b * (R - 1) + (rcb < b ? rcb : rcb - 1));
                    const qb_op_angles& ang = ge.angles[po.op_index];
                    if (ang.slot[0] < 0 && ang.slot2[0] < 0 && ang.cnst[0] == 0.0) {
                        variant |= 32u;  // gamma == 0: m00 = cos(theta / 2) is real
                        // phi == 0 too: m10 = sin(theta / 2) is real (uncontrolled gates only have such bodies)
#if QB_PLAIN_FAST
                        // (only for gates without a control of any kind: those bodies are reached from the op loop directly;
                        //  the rare thread-bit- or externally controlled gate with phi == 0 runs the real-top-left body)
                        if (rcb < 0 && cpos == 31 && extc == 0xff && ang.slot[2] < 0 && ang.slot2[2] < 0 && ang.cnst[2] == 0.0) variant |= 16u;
#else
                        if (rcb < 0 && ang.slot[2] < 0 && ang.slot2[2] < 0 && ang.cnst[2] == 0.0) variant |= 16u;
#endif
                    }
                } else {
                    if (po.tgt_kind == QB_K_THREAD) dpos = po.tgt_pos;
                    else if (po.tgt_kind == QB_K_EXT) extt = po.tgt_pos;
                    if (rcb >= 0) {
                        variant = uint32_t(v_diag_gen<R>());
                        cb = uint32_t(rcb);
                        if (po.tgt_kind == QB_K_REG) treg = 1, tb = po.tgt_pos;
                    } else if (po.tgt_kind == QB_K_REG) {
                        variant = uint32_t(v_diag_reg<R>(0)) + po.tgt_pos;
                    } else {
                        variant = uint32_t(v_diag_out<R>());
                    }
                }
                w = variant | (cpos << 6) | (dpos << 11) | (cb << 17) | (tb << 20) | (treg << 23);
#if QB_PLAIN_FAST
                // bit 31: the commonest op -- a dense gate with a real first column and no control of any kind (variant 48 + b);
                // the op loop reaches its body through one sign test and the two bits of b, without the control test
                if (po.kind == QB_OP_DENSE && (variant ^ 48u) < uint32_t(R)) w |= 0x80000000u;
#endif
                x = extc | (extt << 8);
                if (x != 0xffffu) s_has_ext = 1;
            }
            s_word0[i] = w;
            s_ext[i] = x;
        }
    }
    __syncthreads();  // pass records visible
    uint64_t tile_mask = 0;
#pragma unroll
    for (int i = 0; i < K; ++i) tile_mask |= 1ull << s_sweep.tile_qubits[i];
    for (int p = 0; p < n_pass; ++p) {
        uint32_t e = 0;
#pragma unroll
        for (int b = 0; b < kThreadBits; ++b) e |= ((uint32_t(tid) >> b) & 1u) << s_pass[p].thread_bits[b];
        s_ethr[p * kThreads + tid] = uint16_t(e);
    }
    if (tid < n_pass * R) {
        const int p = tid / R, i = tid % R;
        s_so[p * 8 + i] = swz(1u << s_pass[p].reg_bits[i]) << kAmpShift;
    }
    if (tid < 2 * R) {
        const int which = tid / R, i = tid % R;
        s_gi[which][i] = 1ull << s_sweep.tile_qubits[s_pass[which ? n_pass - 1 : 0].reg_bits[i]];
    }
    // this thread's global-index bits in the first (load) and last (store) pass layouts
    Idx gthr_first = 0, gthr_last = 0;
#pragma unroll
    for (int b = 0; b < kThreadBits; ++b) {
        const Idx bit = Idx((uint32_t(tid) >> b) & 1u);
        gthr_first |= bit << s_sweep.tile_qubits[s_pass[0].thread_bits[b]];
        gthr_last |= bit << s_sweep.tile_qubits[s_pass[n_pass - 1].thread_bits[b]];
    }
    // run number tid scattered over the tile qubits above the QB_LOW_BITS contiguous ones: the 256-byte run this thread prefetches
    Idx pf_off = 0;
#pragma unroll
    for (int b = 0; b < K - QB_LOW_BITS; ++b) pf_off |= Idx((uint32_t(tid) >> b) & 1u) << s_sweep.tile_qubits[QB_LOW_BITS + b];
    const bool l2_prefetch = (flags & QB_SWEEP_L2_PREFETCH) && !product_start && !zero_start && tid < (1 << (K - QB_LOW_BITS));
    // ---- from here on the kernel reads what its predecessors wrote: bound matrices (bind_kernel), the state (previous sweep)
    pdl_wait();
    {
        T* s_mat_t = reinterpret_cast<T*>(s_mat);
        const double* mats = ge.matrices + (size_t(ge.n_ops) + size_t(op_begin)) * 8;
        for (int i = tid; i < n_sop * 8; i += kThreads) s_mat_t[i] = static_cast<T>(ld_cg(mats + i));
        if (product_start) {
            T* s_init_t = reinterpret_cast<T*>(s_init);
            const double* iv = ge.matrices + (size_t(ge.n_ops) + size_t(ge.n_pass_ops)) * 8;
            for (int i = tid; i < 4 * n_eff; i += kThreads) s_init_t[i] = static_cast<T>(ld_cg(iv + i));
            __syncthreads();  // (CTA-uniform branch) the per-thread factor below reads s_init
        }
    }
    // product-state start: factor contributed by this thread's own tile bits (constant over the CTA's tiles)
    C p_thread;
    p_thread.x = T(1), p_thread.y = T(0);
    if (product_start) {
        uint64_t reg_q = 0;
#pragma unroll
        for (int i = 0; i < R; ++i) reg_q |= 1ull << s_sweep.tile_qubits[s_pass[0].reg_bits[i]];
        for (int i = 0; i < K; ++i) {
            const int q = s_sweep.tile_qubits[i];
            if (!((reg_q >> q) & 1ull)) p_thread = cmul<T>(p_thread, s_init[2 * q + int((uint64_t(gthr_first) >> q) & 1ull)]);
        }
        if ((ge.index_offset >> n_eff) != 0) p_thread.x = T(0), p_thread.y = T(0);  // rank bits above the local register start in |0>
    }
    __syncthreads();  // matrices staged
#if QB_PLAIN_FAST
    // plain ops to tangent form in place (their words patched before the per-tile word copy reads them)
    if (tid < 32) stage_tangent<T>(s_mat, s_word0, n_sop, tid, &s_scale);
    __syncthreads();
#endif
    const bool has_ext = s_has_ext != 0;

    C* __restrict__ st = reinterpret_cast<C*>(ge.state);
    const C* __restrict__ src = (sweep_idx == 0 && ge.src_state != nullptr) ? reinterpret_cast<const C*>(ge.src_state) : st;
    const bool do_expect = fuse_expectation && (sweep_idx == ge.n_sweeps - 1) && (ge.diag_table != nullptr);
    const double* __restrict__ table = ge.diag_table;
    const uint64_t index_offset = ge.index_offset;
    const uint64_t not_tile = ~tile_mask & ((n_eff >= 64) ? ~0ull : ((1ull << n_eff) - 1ull));

    // first tile of this CTA: blockIdx.x << m_log2 scattered over the qubits that are not tile bits
    uint64_t base = 0;
    {
        uint64_t t = uint64_t(blockIdx.x) << m_log2;
        for (int q = 0; q < n_eff; ++q)
            if (!((tile_mask >> q) & 1ull)) {
                base |= (t & 1ull) << q;
                t >>= 1;
            }
    }
    const uint32_t n_iter = 1u << m_log2;
    // product-state start: the CTA's tiles differ only in the lowest m_log2 non-tile qubits (`var_mask`); the factor of all
    // other non-tile qubits is the same for every tile of the CTA and joins the per-thread factor once
    uint64_t var_mask = 0;
    if (product_start) {
        uint64_t rest = not_tile;
        for (int i = 0; i < m_log2 && rest; ++i, rest &= rest - 1ull) var_mask |= rest & (0ull - rest);
        for (; rest; rest &= rest - 1ull) {
            const int q = __ffsll((long long)rest) - 1;
            p_thread = cmul<T>(p_thread, s_init[2 * q + int((base >> q) & 1ull)]);
        }
    }
    double acc = 0.0;
    C a[kNReg];

    for (uint32_t it = 0; it < n_iter; ++it, base = ((base | tile_mask) + 1ull) & not_tile) {
        const uint64_t gbase = base | index_offset;
        // ---- per-tile resolution of operands outside the tile (one thread per op)
        const uint32_t* s_w = s_word0;
        if (has_ext) {
            uint32_t* dst = s_word + (it & 1u) * kWordStride;
            if (tid <= n_sop) {
                uint32_t w = s_word0[tid];
                const uint32_t x = s_ext[tid];
                const uint32_t qc = x & 0xffu, qt = (x >> 8) & 0xffu;
                if (qc != 0xffu && !((gbase >> qc) & 1ull)) w = (w & ~(31u << 6)) | (30u << 6);
                if (qt != 0xffu) w |= uint32_t((gbase >> qt) & 1ull) << 16;
                dst[tid] = w;
            }
            s_w = dst;
        }
        // ---- first pass: amplitudes from HBM (or synthesised) straight into registers
        if (product_start) {
            C P = p_thread;
            for (uint64_t v = var_mask; v; v &= v - 1ull) {
                const int q = __ffsll((long long)v) - 1;
                P = cmul<T>(P, s_init[2 * q + int((base >> q) & 1ull)]);
            }
            a[0] = P;
#pragma unroll
            for (int i = 0; i < R; ++i) {
                const int q = 63 - __clzll((long long)s_gi[0][i]);
                const C v0 = s_init[2 * q], v1 = s_init[2 * q + 1];
#pragma unroll
                for (int j = 0; j < (1 << i); ++j) {
                    a[j | (1 << i)] = cmul<T>(a[j], v1);
                    a[j] = cmul<T>(a[j], v0);
                }
            }
        } else {
            Idx ix[kNReg];
            ix[0] = Idx(base) | gthr_first;
#pragma unroll
            for (int i = 0; i < R; ++i)
#pragma unroll
                for (int j = 0; j < (1 << i); ++j) ix[j | (1 << i)] = ix[j] | Idx(s_gi[0][i]);
            if (zero_start) {
#pragma unroll
                for (int j = 0; j < kNReg; ++j) {
                    a[j].x = ((uint64_t(ix[j]) | index_offset) == 0) ? T(1) : T(0);
                    a[j].y = T(0);
                }
            } else {
#pragma unroll
                for (int j = 0; j < kNReg; ++j) a[j] = ld_state(src + ix[j]);
            }
        }
        if (l2_prefetch && it + 1 < n_iter) {
            const uint64_t nb = ((base | tile_mask) + 1ull) & not_tile;
            // per-lane addresses: the bulk form (cp.async.bulk.prefetch.L2 -> UBLKPF) takes a warp-uniform address and would be
            // issued lane by lane; two plain 128-byte line prefetches per 256-byte run cost two instructions per thread
            const char* pf = reinterpret_cast<const char*>(src + (Idx(nb) | pf_off));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(pf));
            if (sizeof(C) == 16) asm volatile("prefetch.global.L2 [%0];" ::"l"(pf + 128));
        }
        // publishes this tile's words; also orders the previous tile's shared-memory reads before this tile's writes
        __syncthreads();

        for (int p = 0; p < n_pass; ++p) {
            const bool last = (p == n_pass - 1);
            const uint32_t e_thr = s_ethr[p * kThreads + tid];
            const uint32_t sb = swz(e_thr) << kAmpShift;
            if (p != 0) {
                uint32_t sx[kNReg];
                sx[0] = sb;
#pragma unroll
                for (int i = 0; i < R; ++i)
#pragma unroll
                    for (int j = 0; j < (1 << i); ++j) sx[j | (1 << i)] = sx[j] ^ s_so[p * 8 + i];
#pragma unroll
                for (int j = 0; j < kNReg; ++j) a[j] = *reinterpret_cast<const C*>(tile_b + sx[j]);
            }

            // ---- gates of this pass, applied in registers ----
            const uint32_t test = e_thr | 0x80000000u;
            const int o_end = s_pass[p].op_end - op_begin;
            int o = s_pass[p].op_begin - op_begin;
            uint32_t word_next = s_w[o];
            for (; o < o_end; ++o) {
                const uint32_t word = word_next;
                word_next = s_w[o + 1];  // prefetch the next dispatch word behind this op's arithmetic
#if QB_PLAIN_FAST
                if (int32_t(word) < 0) {
                    tangent_by_bit<T, R>(word & 3u, a, s_mat + o * 4);
                    continue;
                }
#endif
                if (!((test >> ((word >> 6) & 31u)) & 1u)) continue;
                apply_op<T, R>(word, e_thr, a, s_mat + o * 4);
            }

            // ---- store ----
            if (last) {
#if QB_PLAIN_FAST
                // undo the tangent form's factoring of the sweep's plain ops: every state outside the kernel stays as it was
                const double scale = s_scale;
                if (scale != 1.0) {
#pragma unroll
                    for (int j = 0; j < kNReg; ++j) a[j].x *= T(scale), a[j].y *= T(scale);
                }
#endif
                Idx ix[kNReg];
                ix[0] = Idx(base) | gthr_last;
#pragma unroll
                for (int i = 0; i < R; ++i)
#pragma unroll
                    for (int j = 0; j < (1 << i); ++j) ix[j | (1 << i)] = ix[j] | Idx(s_gi[1][i]);
                if (do_expect) {
                    // fuse_expectation == 2: <H> is all the caller wants (diagonal Hamiltonian): the final state is never read
                    // again and is not written back
#pragma unroll
                    for (int j = 0; j < kNReg; ++j) {
                        if (fuse_expectation != 2) st_state(st + ix[j], a[j]);
                        acc += (double(a[j].x) * double(a[j].x) + double(a[j].y) * double(a[j].y)) * ld_table(table + ix[j]);
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < kNReg; ++j) st_state(st + ix[j], a[j]);
                }
            } else {
                // every thread writes back exactly the shared-memory slots it loaded in this pass: no hazard before the store
                uint32_t sx[kNReg];
                sx[0] = sb;
#pragma unroll
                for (int i = 0; i < R; ++i)
#pragma unroll
                    for (int j = 0; j < (1 << i); ++j) sx[j | (1 << i)] = sx[j] ^ s_so[p * 8 + i];
#pragma unroll
                for (int j = 0; j < kNReg; ++j) *reinterpret_cast<C*>(tile_b + sx[j]) = a[j];
                // the next pass re-reads the tile in its own layout: CTA barrier, unless both passes keep the same tile bits on
                // the warp-index bits -- then every warp only reads what it wrote itself
                if (s_pass[p].flags & QB_PASS_WARP_LOCAL) __syncwarp();
                else __syncthreads();
            }
        }
    }
    if (do_expect) {
        const double total = block_sum(acc, s_red);
        if (tid == 0) ge.partials[blockIdx.x] = total;
    }
}

// ---------------------------------------------------------------------------------------------------
// parameter binding: grid = batch entries
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void bind_matrix(const qb_op_angles& ang, const double* __restrict__ params, double* __restrict__ m) {
    double v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        v[j] = ang.cnst[j] + (ang.slot[j] >= 0 ? ang.coeff[j] * params[ang.slot[j]] : 0.0);
        if (ang.slot2[j] >= 0) v[j] += ang.coeff2[j] * params[ang.slot2[j]];
    }
    const double g = v[0], t = v[1], p = v[2], l = v[3];
    double s, c;
    if (ang.kind == QB_OP_DIAG) {
        sincos(g, &s, &c);
        m[0] = c, m[1] = s, m[2] = 0.0, m[3] = 0.0, m[4] = 0.0, m[5] = 0.0;
        sincos(g + l, &s, &c);
        m[6] = c, m[7] = s;
    } else {
        double sh, ch;
        sincos(0.5 * t, &sh, &ch);
        sincos(g, &s, &c);
        m[0] = c * ch, m[1] = s * ch;
        sincos(g + l, &s, &c);
        m[2] = -c * sh, m[3] = -s * sh;
        sincos(g + p, &s, &c);
        m[4] = c * sh, m[5] = s * sh;
        sincos(g + p + l, &s, &c);
        m[6] = c * ch, m[7] = s * ch;
    }
}

// matrices[0 .. n_ops) by op index (read by the product-state start), matrices[n_ops .. n_ops + n_pass_ops) in pass-op
// order (what a sweep stages: one contiguous, index-free copy)
__global__ void bind_kernel(const BatchEntry* __restrict__ entries) {
    const BatchEntry& en = entries[blockIdx.x];
    for (int o = threadIdx.x; o < en.n_ops; o += blockDim.x) bind_matrix(en.angles[o], en.params, en.matrices + size_t(o) * 8);
    for (int i = threadIdx.x; i < en.n_pass_ops; i += blockDim.x)
        bind_matrix(en.angles[en.pass_ops[i].op_index], en.params, en.matrices + (size_t(en.n_ops) + size_t(i)) * 8);
    // product-state start: per qubit the two amplitudes (re, im, re, im) of its initial single-qubit state
    if (en.init_ops != nullptr) {
        double* init_vec = en.matrices + (size_t(en.n_ops) + size_t(en.n_pass_ops)) * 8;
        for (int q = threadIdx.x; q < en.n_init; q += blockDim.x) {
            double v[4] = {1.0, 0.0, 0.0, 0.0};
            const int op = en.init_ops[q];
            if (op >= 0) {
                double m[8];
                bind_matrix(en.angles[op], en.params, m);
                v[0] = m[0], v[1] = m[1], v[2] = m[4], v[3] = m[5];
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) init_vec[4 * q + i] = v[i];
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// diagonal energies
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ double diag_energy(uint64_t k, const uint64_t* __restrict__ z, const double* __restrict__ c, int n_terms) {
    double e = 0.0;
    for (int t = 0; t < n_terms; ++t) e += (__popcll(k & z[t]) & 1) ? -c[t] : c[t];
    return e;
}

// `accumulate`: add onto the table (term lists longer than the shared-memory staging are built chunk by chunk, in term order)
__global__ void diag_table_kernel(double* __restrict__ table, uint64_t size, uint64_t index_offset,
                                  const uint64_t* __restrict__ z, const double* __restrict__ c, int n_terms, int accumulate) {
    extern __shared__ unsigned char dsm[];
    uint64_t* sz = reinterpret_cast<uint64_t*>(dsm);
    double* sc = reinterpret_cast<double*>(sz + n_terms);
    for (int t = threadIdx.x; t < n_terms; t += blockDim.x) sz[t] = z[t], sc[t] = c[t];
    __syncthreads();
    for (uint64_t k = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; k < size; k += uint64_t(gridDim.x) * blockDim.x) {
        double e = accumulate ? table[k] : 0.0;
        const uint64_t kk = k | index_offset;
        for (int t = 0; t < n_terms; ++t) e += (__popcll(kk & sz[t]) & 1) ? -sc[t] : sc[t];
        table[k] = e;
    }
}

__global__ void diag_lookup_kernel(const uint64_t* __restrict__ states, int64_t n_states, const uint64_t* __restrict__ z,
                                   const double* __restrict__ c, int n_terms, double* __restrict__ out) {
    for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n_states; i += int64_t(gridDim.x) * blockDim.x)
        out[i] = diag_energy(states[i], z, c, n_terms);
}

template <typename T>
__global__ void __launch_bounds__(256)
expect_table_kernel(const typename Cx<T>::type* __restrict__ states, uint64_t state_stride, const double* __restrict__ table, uint64_t size,
                    double* __restrict__ partials, uint64_t partial_stride) {
    __shared__ double s_red[8];
    const auto* state = states + blockIdx.y * state_stride;  // grid.y = batch entry
    double acc = 0.0;
    for (uint64_t k = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; k < size; k += uint64_t(gridDim.x) * blockDim.x) {
        const auto a = state[k];
        acc += (double(a.x) * double(a.x) + double(a.y) * double(a.y)) * table[k];
    }
    const double total = block_sum(acc, s_red);
    if (threadIdx.x == 0) partials[blockIdx.y * partial_stride + blockIdx.x] = total;
}

// One x-mask group of a Pauli sum:  sum_k Re[ psi_k conj(psi_{k^x}) W(k) ],  W(k) = sum_t w_t (-1)^{pc(k & z_t)},
// w_t = coeff_t * i^{#Y_t}.  x == 0 is the diagonal group evaluated on the fly.
template <typename T>
__global__ void __launch_bounds__(256)
expect_group_kernel(const typename Cx<T>::type* __restrict__ states, uint64_t state_stride, uint64_t size, uint64_t index_offset, uint64_t xmask,
                    const uint64_t* __restrict__ z, const double* __restrict__ wr, const double* __restrict__ wi, int n_terms, int stage_terms,
                    double* __restrict__ partials, uint64_t partial_stride) {
    extern __shared__ unsigned char dsm[];
    __shared__ double s_red[8];
    const auto* state = states + blockIdx.y * state_stride;  // grid.y = batch entry
    // terms staged in shared memory while they fit (stage_terms); longer lists are read from global memory (L1 / L2 resident)
    const uint64_t* sz = z;
    const double *swr = wr, *swi = wi;
    if (stage_terms) {
        uint64_t* tz = reinterpret_cast<uint64_t*>(dsm);
        double* twr = reinterpret_cast<double*>(tz + n_terms);
        double* twi = twr + n_terms;
        for (int t = threadIdx.x; t < n_terms; t += blockDim.x) tz[t] = z[t], twr[t] = wr[t], twi[t] = wi[t];
        __syncthreads();
        sz = tz, swr = twr, swi = twi;
    }
    double acc = 0.0;
    for (uint64_t k = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; k < size; k += uint64_t(gridDim.x) * blockDim.x) {
        const auto a = state[k];
        const auto b = xmask ? state[k ^ xmask] : a;
        const double pr = double(a.x) * double(b.x) + double(a.y) * double(b.y);
        const double pi = double(a.y) * double(b.x) - double(a.x) * double(b.y);
        double Wr = 0.0, Wi = 0.0;
        const uint64_t kk = k | index_offset;
        for (int t = 0; t < n_terms; ++t) {
            const bool neg = __popcll(kk & sz[t]) & 1;
            Wr += neg ? -swr[t] : swr[t];
            Wi += neg ? -swi[t] : swi[t];
        }
        acc += pr * Wr - pi * Wi;
    }
    const double total = block_sum(acc, s_red);
    if (threadIdx.x == 0) partials[blockIdx.y * partial_stride + blockIdx.x] = total;
}

// ---------------------------------------------------------------------------------------------------
// tile-fused Pauli-sum expectation (K4): every x-mask group whose flipped qubits fit one tile is evaluated from
// shared memory, so a whole family of groups (e.g. all 24 single-qubit X terms of a transverse-field Ising model in
// three tile sweeps) costs ONE read of the state instead of two reads per group.
//   grid = (tiles, batch entries), block = 256, dynamic smem = 2^kExpTileBits amplitudes
// ---------------------------------------------------------------------------------------------------
constexpr int kExpTileBits = 11;

struct ExpTileSweep {
    int32_t tile_qubits[16];  // kExpTileBits used; first QB_LOW_BITS are qubits 0..QB_LOW_BITS-1
    int32_t group_begin, group_end;
};

struct ExpTileGroup {
    uint32_t xloc;  // x mask in tile-local bit positions
    int32_t term_begin, term_end;
    int32_t trivial;  // 1: single term with z == 0 -> W(k) is the constant (wr, wi) of that term
};

template <typename T>
__global__ void __launch_bounds__(256)
expect_tile_kernel(const typename Cx<T>::type* __restrict__ states, uint64_t state_stride, int n_eff, uint64_t index_offset, ExpTileSweep sw,
                   const ExpTileGroup* __restrict__ groups, const uint64_t* __restrict__ z, const double* __restrict__ wr,
                   const double* __restrict__ wi, double* __restrict__ partials, uint64_t partial_stride) {
    using C = typename Cx<T>::type;
    extern __shared__ __align__(16) unsigned char dsm[];
    C* tile = reinterpret_cast<C*>(dsm);
    __shared__ double s_red[8];
    constexpr int kPerThread = (1 << kExpTileBits) / 256;
    const int tid = threadIdx.x;
    uint64_t tile_mask = 0;
#pragma unroll
    for (int i = 0; i < kExpTileBits; ++i) tile_mask |= 1ull << sw.tile_qubits[i];
    uint64_t base = 0;
    {
        uint64_t t = blockIdx.x;
        for (int q = 0; q < n_eff; ++q)
            if (!((tile_mask >> q) & 1ull)) {
                base |= (t & 1ull) << q;
                t >>= 1;
            }
    }
    // element e = tid + 256 * i : the low 8 tile bits come from tid, the high ones from i
    uint64_t g_lo = 0;
#pragma unroll
    for (int b = 0; b < 8; ++b) g_lo |= uint64_t((tid >> b) & 1) << sw.tile_qubits[b];
    uint64_t g_hi[kPerThread];
#pragma unroll
    for (int i = 0; i < kPerThread; ++i) {
        g_hi[i] = 0;
#pragma unroll
        for (int b = 8; b < kExpTileBits; ++b) g_hi[i] |= uint64_t((i >> (b - 8)) & 1) << sw.tile_qubits[b];
    }
    const C* __restrict__ st = states + blockIdx.y * state_stride;
    C mine[kPerThread];
#pragma unroll
    for (int i = 0; i < kPerThread; ++i) {
        mine[i] = ld_state(st + (base | g_lo | g_hi[i]));
        tile[tid + 256 * i] = mine[i];
    }
    __syncthreads();
    double acc = 0.0;
    for (int g = sw.group_begin; g < sw.group_end; ++g) {
        const ExpTileGroup grp = groups[g];
        if (grp.trivial) {
            // W is one constant (a pure X-type string): Im[psi_k conj(psi_k^x)] is exactly antisymmetric under k <-> k^x, so
            // over the pair it cancels and only the real part counts -- 2 instead of 6 FP64 operations per amplitude
            double s = 0.0;
            const uint32_t hi = grp.xloc >> 8;
            if ((grp.xloc & 255u) == 0u && (hi == 1u || hi == 2u || hi == 4u)) {
                // the flipped bit is one of the thread's own element bits: both partners sit in this thread's registers --
                // no shared-memory read, and each pair is visited once (counted twice)
#define QB_PAIRS(S)                                                                                                    \
    _Pragma("unroll") for (int i = 0; i < kPerThread; ++i) if (!(i & S))                                                \
        s = fma(double(mine[i].x), double(mine[i | S].x), fma(double(mine[i].y), double(mine[i | S].y), s));
                if (hi == 1u) { QB_PAIRS(1) } else if (hi == 2u) { QB_PAIRS(2) } else { QB_PAIRS(4) }
#undef QB_PAIRS
                s += s;
            } else {
#pragma unroll
                for (int i = 0; i < kPerThread; ++i) {
                    const C a = mine[i];
                    const C b = tile[(tid + 256 * i) ^ grp.xloc];
                    s = fma(double(a.x), double(b.x), fma(double(a.y), double(b.y), s));
                }
            }
            acc = fma(wr[grp.term_begin], s, acc);
            continue;
        }
#pragma unroll
        for (int i = 0; i < kPerThread; ++i) {
            const C a = mine[i];
            const C b = tile[(tid + 256 * i) ^ grp.xloc];
            const double pr = double(a.x) * double(b.x) + double(a.y) * double(b.y);
            const double pi = double(a.y) * double(b.x) - double(a.x) * double(b.y);
            double Wr = 0.0, Wi = 0.0;
            const uint64_t kk = base | g_lo | g_hi[i] | index_offset;
            for (int t = grp.term_begin; t < grp.term_end; ++t) {
                const bool neg = __popcll(kk & z[t]) & 1;
                Wr += neg ? -wr[t] : wr[t];
                Wi += neg ? -wi[t] : wi[t];
            }
            acc += pr * Wr - pi * Wi;
        }
    }
    const double total = block_sum(acc, s_red);
    if (tid == 0) partials[blockIdx.y * partial_stride + blockIdx.x] = total;
}

// out[b] (+)= sum_i partials[b * stride + i]  in a fixed order (deterministic).
__global__ void __launch_bounds__(256)
reduce_partials_kernel(const double* partials, int64_t stride, int64_t count, double* out, int accumulate) {
    __shared__ double s_red[8];
    pdl_launch_dependents();
    pdl_wait();
    const double* p = partials + blockIdx.x * stride;
    double acc = 0.0;
    for (int64_t i = threadIdx.x; i < count; i += blockDim.x) acc += ld_cg(p + i);
    const double total = block_sum(acc, s_red);
    if (threadIdx.x == 0) out[blockIdx.x] = accumulate ? out[blockIdx.x] + total : total;
}

// ---------------------------------------------------------------------------------------------------
// term-resolved expectation (qb_evaluate_observables): <P_t> of every distinct Pauli string P_t = i^{#Y} X^x Z^z of a set of
// observables, one value per string, from one read of the state per tile sweep of x-mask groups.  With the pair product
// p_k = psi_k conj(psi_{k^x}):   <P_t> = sign_t * sum_k (-1)^{pc(k & z_t)} * (#Y_t odd ? Im p_k : Re p_k),
// sign_t = -1 for #Y = 1, 2 (mod 4), +1 otherwise (applied by reduce_term_partials_kernel).  Every CTA writes one partial per
// (term, CTA); the second stage sums them in a fixed order: no atomics, and a term's value depends on neither the other terms
// of its launch nor the batch it is evaluated in.
// ---------------------------------------------------------------------------------------------------
constexpr int kTermChunk = 8;  // accumulators held in registers per pass over the thread's amplitudes

struct TermGroup {
    uint64_t xmask;     // flipped qubits
    uint32_t xloc;      // x mask in tile-local bit positions (tile sweeps)
    int32_t term_begin, term_end;
    int32_t real_only;  // no string of the group has an odd number of Y: Im p_k is never read
};

// block reduction of kTermChunk accumulators (fixed tree per term); thread c < nc writes term c's CTA total to out[c * stride]
__device__ __forceinline__ void term_chunk_store(double (&acc)[kTermChunk], int nc, double* s_red, double* __restrict__ out, uint64_t stride) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int c = 0; c < kTermChunk; ++c) {
        const double v = warp_sum(acc[c]);
        if (lane == 0) s_red[warp * kTermChunk + c] = v;
    }
    __syncthreads();
    if (threadIdx.x < nc) {
        const int nw = blockDim.x >> 5;
        double total = 0.0;
        for (int w = 0; w < nw; ++w) total += s_red[w * kTermChunk + threadIdx.x];
        out[threadIdx.x * stride] = total;
    }
    __syncthreads();
}

// terms [lo, hi) of one group over the thread's kPerThread pair products; kk[i] = global index of amplitude i
template <int kPerThread>
__device__ __forceinline__ void term_chunks(const double (&pr)[kPerThread], const double (&pi)[kPerThread], const uint64_t (&kk)[kPerThread],
                                            const uint64_t* __restrict__ z, const int8_t* __restrict__ im, int lo, int hi, int t0,
                                            double* s_red, double* __restrict__ part, uint64_t count) {
    for (int c0 = lo; c0 < hi; c0 += kTermChunk) {
        const int nc = min(kTermChunk, hi - c0);
        uint64_t zc[kTermChunk];
        uint32_t ic = 0;  // bit c: term c reads Im p_k
        double acc[kTermChunk];
#pragma unroll
        for (int c = 0; c < kTermChunk; ++c) {
            zc[c] = c < nc ? z[c0 + c] : 0;
            ic |= (c < nc && im[c0 + c] != 0) ? 1u << c : 0u;
            acc[c] = 0.0;
        }
#pragma unroll
        for (int i = 0; i < kPerThread; ++i)
#pragma unroll
            for (int c = 0; c < kTermChunk; ++c) {
                const double v = ((ic >> c) & 1u) ? pi[i] : pr[i];
                acc[c] += (__popcll(kk[i] & zc[c]) & 1) ? -v : v;
            }
        term_chunk_store(acc, nc, s_red, part + uint64_t(c0 - t0) * count, count);
    }
}

// grid = (tiles, batch entries), block = 256, dynamic smem = 2^kExpTileBits amplitudes.  Terms [t0, t1) of the sweep's groups;
// partials[((entry * (t1 - t0)) + t - t0) * tiles + tile].
template <typename T>
__global__ void __launch_bounds__(256)
expect_terms_tile_kernel(const typename Cx<T>::type* __restrict__ states, uint64_t state_stride, int n_eff, ExpTileSweep sw,
                         const TermGroup* __restrict__ groups, const uint64_t* __restrict__ z, const int8_t* __restrict__ im, int t0, int t1,
                         double* __restrict__ partials) {
    using C = typename Cx<T>::type;
    extern __shared__ __align__(16) unsigned char dsm[];
    C* tile = reinterpret_cast<C*>(dsm);
    __shared__ double s_red[8 * kTermChunk];
    constexpr int kPerThread = (1 << kExpTileBits) / 256;
    const int tid = threadIdx.x;
    uint64_t tile_mask = 0;
#pragma unroll
    for (int i = 0; i < kExpTileBits; ++i) tile_mask |= 1ull << sw.tile_qubits[i];
    uint64_t base = 0;
    {
        uint64_t t = blockIdx.x;
        for (int q = 0; q < n_eff; ++q)
            if (!((tile_mask >> q) & 1ull)) {
                base |= (t & 1ull) << q;
                t >>= 1;
            }
    }
    // element e = tid + 256 * i : the low 8 tile bits come from tid, the high ones from i
    uint64_t g_lo = 0;
#pragma unroll
    for (int b = 0; b < 8; ++b) g_lo |= uint64_t((tid >> b) & 1) << sw.tile_qubits[b];
    uint64_t kk[kPerThread];
#pragma unroll
    for (int i = 0; i < kPerThread; ++i) {
        kk[i] = base | g_lo;
#pragma unroll
        for (int b = 8; b < kExpTileBits; ++b) kk[i] |= uint64_t((i >> (b - 8)) & 1) << sw.tile_qubits[b];
    }
    const C* __restrict__ st = states + blockIdx.y * state_stride;
    C mine[kPerThread];
#pragma unroll
    for (int i = 0; i < kPerThread; ++i) {
        mine[i] = ld_state(st + kk[i]);
        tile[tid + 256 * i] = mine[i];
    }
    __syncthreads();
    const uint64_t count = gridDim.x;
    double* part = partials + uint64_t(blockIdx.y) * uint64_t(t1 - t0) * count + blockIdx.x;
    for (int g = sw.group_begin; g < sw.group_end; ++g) {
        const TermGroup grp = groups[g];
        const int lo = max(grp.term_begin, t0), hi = min(grp.term_end, t1);
        if (lo >= hi) continue;
        double pr[kPerThread], pi[kPerThread];
        const uint32_t hi_bits = grp.xloc >> 8;
        if (grp.xloc == 0u) {
            // diagonal group: p_k = |psi_k|^2
#pragma unroll
            for (int i = 0; i < kPerThread; ++i) {
                pr[i] = fma(double(mine[i].x), double(mine[i].x), double(mine[i].y) * double(mine[i].y));
                pi[i] = 0.0;
            }
        } else if (grp.real_only && (grp.xloc & 255u) == 0u && (hi_bits == 1u || hi_bits == 2u || hi_bits == 4u)) {
            // the flipped bit is one of the thread's own element bits: the partner sits in this thread's registers (no
            // shared-memory read), and only the real part of the pair product is needed
#define QB_REG_PAIRS(S)                                                                                                \
    _Pragma("unroll") for (int i = 0; i < kPerThread; ++i) {                                                            \
        pr[i] = fma(double(mine[i].x), double(mine[i ^ S].x), double(mine[i].y) * double(mine[i ^ S].y));               \
        pi[i] = 0.0;                                                                                                    \
    }
            if (hi_bits == 1u) { QB_REG_PAIRS(1) } else if (hi_bits == 2u) { QB_REG_PAIRS(2) } else { QB_REG_PAIRS(4) }
#undef QB_REG_PAIRS
        } else {
#pragma unroll
            for (int i = 0; i < kPerThread; ++i) {
                const C a = mine[i];
                const C b = tile[(tid + 256 * i) ^ grp.xloc];
                pr[i] = fma(double(a.x), double(b.x), double(a.y) * double(b.y));
                pi[i] = grp.real_only ? 0.0 : fma(double(a.y), double(b.x), -double(a.x) * double(b.y));
            }
        }
        term_chunks(pr, pi, kk, z, im, lo, hi, t0, s_red, part, count);
    }
}

// One group whose x mask does not fit a tile: two reads of the state per chunk of kTermChunk terms.
// grid = (blocks, batch entries), block = 256; terms [lo, hi) of the group, partials as above with count = blocks.
template <typename T>
__global__ void __launch_bounds__(256)
expect_terms_group_kernel(const typename Cx<T>::type* __restrict__ states, uint64_t state_stride, uint64_t size, uint64_t xmask,
                          const uint64_t* __restrict__ z, const int8_t* __restrict__ im, int lo, int hi, int t0, int nt,
                          double* __restrict__ partials) {
    __shared__ double s_red[8 * kTermChunk];
    const auto* state = states + blockIdx.y * state_stride;
    const uint64_t count = gridDim.x;
    double* part = partials + uint64_t(blockIdx.y) * uint64_t(nt) * count + blockIdx.x;
    for (int c0 = lo; c0 < hi; c0 += kTermChunk) {
        const int nc = min(kTermChunk, hi - c0);
        uint64_t zc[kTermChunk];
        uint32_t ic = 0;  // bit c: term c reads Im p_k
        double acc[kTermChunk];
#pragma unroll
        for (int c = 0; c < kTermChunk; ++c) {
            zc[c] = c < nc ? z[c0 + c] : 0;
            ic |= (c < nc && im[c0 + c] != 0) ? 1u << c : 0u;
            acc[c] = 0.0;
        }
        for (uint64_t k = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; k < size; k += uint64_t(gridDim.x) * blockDim.x) {
            const auto a = state[k];
            const auto b = state[k ^ xmask];
            const double pr = fma(double(a.x), double(b.x), double(a.y) * double(b.y));
            const double pi = fma(double(a.y), double(b.x), -double(a.x) * double(b.y));
#pragma unroll
            for (int c = 0; c < kTermChunk; ++c) {
                const double v = ((ic >> c) & 1u) ? pi : pr;
                acc[c] += (__popcll(k & zc[c]) & 1) ? -v : v;
            }
        }
        term_chunk_store(acc, nc, s_red, part + uint64_t(c0 - t0) * count, count);
    }
}

// terms[entry * terms_stride + t0 + t] = sign[t0 + t] * sum_i partials[(entry * nt + t) * count + i]  (fixed order)
// grid = (nt, batch entries)
__global__ void __launch_bounds__(256)
reduce_term_partials_kernel(const double* __restrict__ partials, int64_t count, int nt, const double* __restrict__ sign, int t0,
                            double* __restrict__ terms, int64_t terms_stride) {
    __shared__ double s_red[8];
    const double* p = partials + (int64_t(blockIdx.y) * nt + blockIdx.x) * count;
    double acc = 0.0;
    for (int64_t i = threadIdx.x; i < count; i += blockDim.x) acc += p[i];
    const double total = block_sum(acc, s_red);
    if (threadIdx.x == 0) terms[blockIdx.y * terms_stride + t0 + blockIdx.x] = sign[t0 + blockIdx.x] * total;
}

// out[entry * n_obs + j] = sum_e coeff[e] * terms[entry * n_terms + cols[e]] over row j's entries (ascending term order)
// grid = (ceil(n_obs / 128), batch entries), block = 128
__global__ void __launch_bounds__(128)
combine_observables_kernel(const double* __restrict__ terms, int n_terms, const int64_t* __restrict__ row_begin,
                           const int32_t* __restrict__ cols, const double* __restrict__ coeff, int n_obs, double* __restrict__ out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_obs) return;
    const double* t = terms + int64_t(blockIdx.y) * n_terms;
    double s = 0.0;
    for (int64_t e = row_begin[j]; e < row_begin[j + 1]; ++e) s = fma(coeff[e], t[cols[e]], s);
    out[int64_t(blockIdx.y) * n_obs + j] = s;
}

// ---------------------------------------------------------------------------------------------------
// sampling: |psi|^2 chunk sums -> inclusive scan of chunk sums -> per-shot two-level search
// ---------------------------------------------------------------------------------------------------
constexpr int kChunkBits = 9;  // 512 amplitudes per chunk
constexpr int kChunk = 1 << kChunkBits;

// grid.x covers chunks (one warp per chunk), grid.y = batch entry; states are `state_stride` amplitudes apart
template <typename T>
__global__ void __launch_bounds__(256)
chunk_prob_kernel(const typename Cx<T>::type* __restrict__ states, uint64_t state_stride, uint64_t n_chunks,
                  double* __restrict__ chunk_sums) {
    const int lane = threadIdx.x & 31;
    const uint64_t warps_per_grid = uint64_t(gridDim.x) * (blockDim.x >> 5);
    const auto* st = states + blockIdx.y * state_stride;
    double* out = chunk_sums + blockIdx.y * n_chunks;
    for (uint64_t ch = blockIdx.x * uint64_t(blockDim.x >> 5) + (threadIdx.x >> 5); ch < n_chunks; ch += warps_per_grid) {
        double acc = 0.0;
#pragma unroll
        for (int i = 0; i < kChunk / 32; ++i) {
            const auto a = st[ch * kChunk + i * 32 + lane];
            acc += double(a.x) * double(a.x) + double(a.y) * double(a.y);
        }
        acc = warp_sum(acc);
        if (lane == 0) out[ch] = acc;
    }
}

// in-place inclusive scan of n_chunks doubles per batch entry; one CTA of 1024 threads per entry
__global__ void __launch_bounds__(1024)
scan_chunks_kernel(double* __restrict__ chunk_sums, uint64_t n_chunks) {
    __shared__ double s_tot[1024];
    double* data = chunk_sums + blockIdx.x * n_chunks;
    const uint64_t per = (n_chunks + blockDim.x - 1) / blockDim.x;
    const uint64_t lo = threadIdx.x * per, hi = (lo + per < n_chunks) ? lo + per : n_chunks;
    double acc = 0.0;
    for (uint64_t i = lo; i < hi; ++i) acc += data[i];
    s_tot[threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double run = 0.0;
        for (int i = 0; i < int(blockDim.x); ++i) {
            const double v = s_tot[i];
            s_tot[i] = run;
            run += v;
        }
    }
    __syncthreads();
    double run = s_tot[threadIdx.x];
    for (uint64_t i = lo; i < hi; ++i) {
        run += data[i];
        data[i] = run;
    }
}

// one warp per shot: index = first k with cdf(k) / total > u   (searchsorted(cdf / cdf[-1], u, side='right'))
// searchsorted never returns an index of probability zero for u < 1 (such an entry repeats its predecessor's cdf).  The warp
// scan below sums in tree order, so at a cdf boundary a zero-probability lane can see a larger running sum than the non-zero
// lane before it: only lanes with pr > 0 may be hits, and the fallback for a chunk whose running sum misses u by rounding is
// its last entry with pr > 0.
template <typename T>
__global__ void __launch_bounds__(256)
sample_kernel(const typename Cx<T>::type* __restrict__ states, uint64_t state_stride, const double* __restrict__ chunk_cdf,
              uint64_t n_chunks, uint64_t valid_size, const double* __restrict__ uniforms, int shots, int64_t* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int shot = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (shot >= shots) return;
    const auto* st = states + blockIdx.y * state_stride;
    const double* cdf = chunk_cdf + blockIdx.y * n_chunks;
    const double total = cdf[n_chunks - 1];
    const double u = uniforms[blockIdx.y * uint64_t(shots) + shot];
    // first chunk whose inclusive cdf / total exceeds u
    uint64_t lo = 0, hi = n_chunks - 1;
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if (cdf[mid] / total > u) hi = mid;
        else lo = mid + 1;
    }
    double run = lo ? cdf[lo - 1] : 0.0;
    int64_t found = -1, last_nz = -1;
    for (int i = 0; i < kChunk / 32 && found < 0; ++i) {
        const uint64_t k = lo * kChunk + i * 32 + lane;
        const auto a = st[k];
        const double pr = double(a.x) * double(a.x) + double(a.y) * double(a.y);
        double inc = pr;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double nb = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += nb;
        }
        const bool hit = pr > 0.0 && ((run + inc) / total > u);
        const unsigned ballot = __ballot_sync(0xffffffffu, hit);
        const unsigned nonzero = __ballot_sync(0xffffffffu, pr > 0.0);
        if (ballot) found = int64_t(lo * kChunk + i * 32 + (__ffs(ballot) - 1));
        else if (nonzero) last_nz = int64_t(lo * kChunk + i * 32 + (31 - __clz(nonzero)));
        run += __shfl_sync(0xffffffffu, inc, 31);
    }
    if (found < 0) found = last_nz;  // rounding at the very top of a chunk
    if (found < 0) found = int64_t(lo * kChunk + kChunk - 1);  // (no mass in the chunk: only for u outside [0, 1))
    if (uint64_t(found) >= valid_size) found = int64_t(valid_size - 1);
    if (lane == 0) out[blockIdx.y * uint64_t(shots) + shot] = found;
}

// ---------------------------------------------------------------------------------------------------
// exact CVaR(alpha) of a diagonal Hamiltonian (K6): the lower alpha-tail of |psi_k|^2 in (E(k), k) order, weighted by E(k)
// (expectation.lower_tail_expectation_arrays on the full distribution).  `perm` = sorted position -> basis index and
// `energy` = E at each sorted position (the Hamiltonian's order data); perm == nullptr walks basis order with energy = E(k)
// (the unsorted greedy rule of alpha ~ 1).  chunk sums -> scan_chunks_kernel on both sums -> one warp per entry finishes.
// Every sum runs in a fixed order (lane, then warp_sum / warp scan): bit-identical across runs and batch compositions.
// ---------------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ double cvar_prob(const typename Cx<T>::type* __restrict__ st, const uint32_t* __restrict__ perm, uint64_t pos) {
    const auto a = st[perm ? uint64_t(perm[pos]) : pos];
    return double(a.x) * double(a.x) + double(a.y) * double(a.y);
}

// grid.x covers chunks (one warp per 512 sorted positions), grid.y = batch entry: chunk mass and chunk sum p * E
template <typename T>
__global__ void __launch_bounds__(256)
cvar_chunk_kernel(const typename Cx<T>::type* __restrict__ states, uint64_t state_stride, const uint32_t* __restrict__ perm,
                  const double* __restrict__ energy, uint64_t n_chunks, double* __restrict__ chunk_mass, double* __restrict__ chunk_pe) {
    const int lane = threadIdx.x & 31;
    const uint64_t warps_per_grid = uint64_t(gridDim.x) * (blockDim.x >> 5);
    const auto* st = states + blockIdx.y * state_stride;
    for (uint64_t ch = blockIdx.x * uint64_t(blockDim.x >> 5) + (threadIdx.x >> 5); ch < n_chunks; ch += warps_per_grid) {
        double m = 0.0, s = 0.0;
#pragma unroll 4
        for (int i = 0; i < kChunk / 32; ++i) {
            const uint64_t pos = ch * kChunk + i * 32 + lane;
            const double p = cvar_prob<T>(st, perm, pos);
            m += p;
            s = fma(p, energy[pos], s);
        }
        m = warp_sum(m);
        s = warp_sum(s);
        if (lane == 0) chunk_mass[blockIdx.y * n_chunks + ch] = m, chunk_pe[blockIdx.y * n_chunks + ch] = s;
    }
}

__global__ void iota_u32_kernel(uint32_t* __restrict__ out, uint64_t size) {
    for (uint64_t k = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; k < size; k += uint64_t(gridDim.x) * blockDim.x) out[k] = uint32_t(k);
}

// one warp per batch entry; mass_cdf / pe_cdf are the inclusive scans of the chunk sums.  The stop entry is the first k whose running
// mass reaches alpha - (atol + rtol * alpha) (numpy.isclose); out = (sum_{i<k} p_i E_i + min(alpha - cum_{k-1}, p_k) E_k) / alpha.
template <typename T>
__global__ void __launch_bounds__(256)
cvar_finish_kernel(const typename Cx<T>::type* __restrict__ states, uint64_t state_stride, const uint32_t* __restrict__ perm,
                   const double* __restrict__ energy, const double* __restrict__ mass_cdf, const double* __restrict__ pe_cdf, uint64_t n_chunks,
                   double alpha, int batch, double* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int entry = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (entry >= batch) return;
    const auto* st = states + entry * state_stride;
    const double* cdf = mass_cdf + entry * n_chunks;
    const double* pcdf = pe_cdf + entry * n_chunks;
    const double bound = alpha - (1e-8 + 1e-5 * alpha);
    if (cdf[n_chunks - 1] < bound) {  // the whole distribution weighs less than the bound: every entry is taken
        if (lane == 0) out[entry] = pcdf[n_chunks - 1] / alpha;
        return;
    }
    uint64_t lo = 0, hi = n_chunks - 1;
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if (cdf[mid] >= bound) hi = mid;
        else lo = mid + 1;
    }
    double run = lo ? cdf[lo - 1] : 0.0, acc = lo ? pcdf[lo - 1] : 0.0;
    for (int i = 0; i < kChunk / 32; ++i) {
        const uint64_t pos = lo * kChunk + i * 32 + lane;
        const double p = cvar_prob<T>(st, perm, pos);
        const double e = energy[pos];
        double inc = p, pe = p * e;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double nb = __shfl_up_sync(0xffffffffu, inc, o);
            const double nbe = __shfl_up_sync(0xffffffffu, pe, o);
            if (lane >= o) inc += nb, pe += nbe;
        }
        // the last entry of the chunk stops the walk when the in-chunk running sum misses the bound by rounding only
        const bool hit = run + inc >= bound || (i == kChunk / 32 - 1 && lane == 31);
        const unsigned ballot = __ballot_sync(0xffffffffu, hit);
        const double excl = __shfl_up_sync(0xffffffffu, inc, 1), excl_pe = __shfl_up_sync(0xffffffffu, pe, 1);
        if (ballot) {
            if (lane == __ffs(ballot) - 1) {
                const double before = run + (lane ? excl : 0.0);
                out[entry] = (acc + (lane ? excl_pe : 0.0) + fmin(alpha - before, p) * e) / alpha;
            }
            return;
        }
        run += __shfl_sync(0xffffffffu, inc, 31);
        acc += __shfl_sync(0xffffffffu, pe, 31);
    }
}

// ---------------------------------------------------------------------------------------------------
// exact CVaR(alpha) of a SHARDED state (K8): one radix-digit pass of a sort-free weighted selection over one shard.
// The stable ascending (E(k), logical k) order is the order of the composite key (energy_key(E(k)), logical k); the stop entry
// of the greedy fill is the smallest key whose inclusive mass reaches the bound.  The host fixes the key digit by digit: every
// pass histograms, over the entries that match the prefix fixed so far, the next digit -- per bucket the mass, sum p * E, the
// count, min / max of the energy key and the least physical index -- and the host keeps the bucket in which the bound falls.
//   digit_kind 0: bits [e_free - bits, e_free) of the energy key;  1: logical index bits, read from physical positions pos[]
// Determinism: per warp and iteration the entries of one digit are summed by their lowest lane in lane order, the per-warp
// histograms are added in warp order, and per-CTA partials are reduced in CTA order (cvar_select_reduce_kernel).  Count, min
// and max are integers (atomics are order-free).  cache_mode 1 writes (p, E) of every entry into `cache` (the spare shard
// buffer, 16 B per amplitude), mode 2 reads them from there instead of the state and the Hamiltonian.
// ---------------------------------------------------------------------------------------------------
constexpr int kSelBits = 8;
constexpr int kSelBuckets = 1 << kSelBits;
constexpr int kSelWarps = 8;

struct SelectArgs {
    uint64_t e_prefix;             // fixed high bits of the energy key (its low e_free bits are open)
    uint64_t idx_mask, idx_value;  // physical index bits fixed by the logical-index prefix
    int32_t e_free;                // 64: no energy constraint (alpha ~ 1 orders by the logical index alone)
    int32_t digit_kind, bits;
    int32_t pos[kSelBits];         // index digit: physical positions of its logical bits, lowest first
};

// order-preserving 64-bit key of a double; -0.0 gets the key of +0.0 (radix sort / numpy stable argsort treat them as tied)
__device__ __forceinline__ uint64_t energy_key(double e) {
    uint64_t u = uint64_t(__double_as_longlong(e));
    if (u == 0x8000000000000000ull) u = 0;
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}

// Whether an entry with value key `key` (the energy key here, the probability key in top_select_kernel) and physical index kk
// matches the prefix of `a`, and the digit d of its key (digit_kind 0) or of its logical index (digit_kind 1) for this pass
__device__ __forceinline__ bool select_digit(const SelectArgs& a, uint64_t key, uint64_t kk, unsigned& d) {
    const bool ok = (kk & a.idx_mask) == a.idx_value && (a.e_free >= 64 || (key >> a.e_free) == a.e_prefix);
    d = 0;
    if (a.digit_kind == 0) {
        d = unsigned(key >> (a.e_free - a.bits)) & ((1u << a.bits) - 1u);
    } else {
#pragma unroll
        for (int j = 0; j < kSelBits; ++j)  // (unrolled: constant indices keep a.pos in registers, off the stack)
            if (j < a.bits) d |= unsigned((kk >> a.pos[j]) & 1) << j;
    }
    return ok;
}

// grid = n_cta (fixed by the device and the shard size), block = 32 * kSelWarps.  part_* = [bucket][cta];
// ints = [count | emin | emax | kmin][bucket], initialised by the caller (0, ~0, 0, ~0)
template <typename T>
__global__ void __launch_bounds__(32 * kSelWarps)
cvar_select_kernel(const typename Cx<T>::type* __restrict__ state, double2* __restrict__ cache, int cache_mode, uint64_t size,
                   uint64_t index_offset, const uint64_t* __restrict__ z, const double* __restrict__ c, int n_terms, SelectArgs a,
                   double* __restrict__ part_mass, double* __restrict__ part_pe, unsigned long long* __restrict__ ints) {
    __shared__ double h_m[kSelWarps][kSelBuckets], h_s[kSelWarps][kSelBuckets];
    __shared__ double st_p[kSelWarps][32], st_e[kSelWarps][32];
    __shared__ unsigned long long st_k[kSelWarps][32];
    __shared__ unsigned long long s_cnt[kSelBuckets], s_min[kSelBuckets], s_max[kSelBuckets], s_kmin[kSelBuckets];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int b = threadIdx.x; b < kSelBuckets; b += blockDim.x) {
        for (int w = 0; w < kSelWarps; ++w) h_m[w][b] = 0.0, h_s[w][b] = 0.0;
        s_cnt[b] = 0, s_min[b] = ~0ull, s_max[b] = 0, s_kmin[b] = ~0ull;
    }
    __syncthreads();
    const uint64_t stride = uint64_t(gridDim.x) * kSelWarps * 32;
    // size is a multiple of 32: every lane of a warp runs the same iterations (the warp-synchronous steps below need it)
    for (uint64_t k = (uint64_t(blockIdx.x) * kSelWarps + warp) * 32 + lane; k < size; k += stride) {
        double p, e;
        if (cache_mode == 2) {
            const double2 v = cache[k];
            p = v.x, e = v.y;
        } else {
            const auto amp = state[k];
            p = double(amp.x) * double(amp.x) + double(amp.y) * double(amp.y);
            e = 0.0;  // diag_table_kernel's loop: the same double, so ties are the ones the single-GPU route sees
            const uint64_t kk = k | index_offset;
            for (int t = 0; t < n_terms; ++t) e += (__popcll(kk & z[t]) & 1) ? -c[t] : c[t];
            if (cache_mode == 1) cache[k] = make_double2(p, e);
        }
        const uint64_t kk = k | index_offset;
        unsigned d;
        const bool ok = select_digit(a, energy_key(e), kk, d);
        const unsigned peers = __match_any_sync(0xffffffffu, ok ? d : 0xffffffffu);
        st_p[warp][lane] = p, st_e[warp][lane] = e, st_k[warp][lane] = kk;
        __syncwarp();
        if (ok && lane == __ffs(peers) - 1) {  // the lowest lane of every digit sums its peers in lane order
            double m = 0.0, s = 0.0;
            uint64_t lo = ~0ull, hi = 0, kmin = ~0ull;
            for (unsigned rest = peers; rest; rest &= rest - 1) {
                const int l = __ffs(rest) - 1;
                const double pl = st_p[warp][l], el = st_e[warp][l];
                const uint64_t kl = energy_key(el);
                m += pl, s += pl * el;
                lo = kl < lo ? kl : lo, hi = kl > hi ? kl : hi;
                kmin = st_k[warp][l] < kmin ? st_k[warp][l] : kmin;
            }
            h_m[warp][d] += m, h_s[warp][d] += s;
            atomicAdd(&s_cnt[d], (unsigned long long)__popc(peers));
            atomicMin(&s_min[d], (unsigned long long)lo);
            atomicMax(&s_max[d], (unsigned long long)hi);
            atomicMin(&s_kmin[d], (unsigned long long)kmin);
        }
        __syncwarp();
    }
    __syncthreads();
    for (int b = threadIdx.x; b < kSelBuckets; b += blockDim.x) {
        double m = 0.0, s = 0.0;
        for (int w = 0; w < kSelWarps; ++w) m += h_m[w][b], s += h_s[w][b];
        part_mass[uint64_t(b) * gridDim.x + blockIdx.x] = m;
        part_pe[uint64_t(b) * gridDim.x + blockIdx.x] = s;
        if (s_cnt[b]) {
            atomicAdd(&ints[b], s_cnt[b]);
            atomicMin(&ints[kSelBuckets + b], s_min[b]);
            atomicMax(&ints[2 * kSelBuckets + b], s_max[b]);
            atomicMin(&ints[3 * kSelBuckets + b], s_kmin[b]);
        }
    }
}

// out[row] = sum over CTAs (in CTA order, then block_sum's fixed tree) of part[row * n_cta + i];  grid = 2 * kSelBuckets rows
__global__ void __launch_bounds__(256)
cvar_select_reduce_kernel(const double* __restrict__ part, int n_cta, double* __restrict__ out) {
    __shared__ double s_red[8];
    const double* p = part + uint64_t(blockIdx.x) * n_cta;
    double acc = 0.0;
    for (int i = threadIdx.x; i < n_cta; i += blockDim.x) acc += p[i];
    const double total = block_sum(acc, s_red);
    if (threadIdx.x == 0) out[blockIdx.x] = total;
}

// ---------------------------------------------------------------------------------------------------
// most probable basis states (K9): the max_states first entries of the composite key (prob_key(p_k), logical k) -- descending
// p_k, ties in ascending logical index -- among the entries with p_k > 0 and p_k >= min_probability, without sorting the state.
// top_select_kernel histograms one 8-bit digit of that key per pass (counts only, over the entries matching the prefix fixed so
// far; SelectArgs / select_digit of the CVaR select with the probability key in place of the energy key); the host picks the
// bucket (qb_top_select_pick) until the stop key is known, then top_collect_kernel writes every entry up to the stop key.
// p_k = re^2 + im^2 in double, rounded without FMA contraction, so a NumPy re * re + im * im on the same amplitudes gives
// every bit.  Counts are integers: the histograms and the compaction are the same on every run whatever the scheduling.
// ---------------------------------------------------------------------------------------------------
struct TopSelectArgs {
    SelectArgs sel;  // prefix and digit of this pass (e_prefix / e_free: the probability key's)
    double min_probability;
    int32_t entry;   // row of `states`
};

struct TopCollectArgs {
    uint64_t stop_key, stop_index;  // every eligible entry with (prob_key, logical k) <= (stop_key, stop_index) is written
    double min_probability;
    int32_t entry;                  // row of `states`
    int32_t n_pos;                  // 0: logical index == physical index; else logical bit q sits at physical position pos[q]
    int8_t pos[64];
};

template <typename C>
__device__ __forceinline__ double top_prob(C a) {
    const double x = double(a.x), y = double(a.y);
    return __dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y));
}

// ascending key = descending p: for p > 0 the bit pattern is ordered like the value
__device__ __forceinline__ uint64_t prob_key(double p) { return ~uint64_t(__double_as_longlong(p)); }

__device__ __forceinline__ bool top_eligible(double p, double min_probability) { return p > 0.0 && p >= min_probability; }

constexpr int kTopUnroll = 4;  // amplitudes loaded per thread before any is processed

// grid = (n_cta, entries of this pass), block = 32 * kSelWarps; counts = [entry][bucket], zeroed by the caller.  Idx: uint32_t
// up to 2^31 amplitudes, uint64_t above (the sweep kernels' switch).
template <typename T, typename Idx>
__global__ void __launch_bounds__(32 * kSelWarps)
top_select_kernel(const typename Cx<T>::type* __restrict__ states, uint64_t state_stride, Idx size, uint64_t index_offset,
                  const TopSelectArgs* __restrict__ args, unsigned long long* __restrict__ counts) {
    __shared__ uint32_t h[kSelWarps][kSelBuckets];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int b = threadIdx.x; b < kSelWarps * kSelBuckets; b += blockDim.x) h[b / kSelBuckets][b % kSelBuckets] = 0;
    __syncthreads();
    const TopSelectArgs ta = args[blockIdx.y];
    const auto* st = states + uint64_t(ta.entry) * state_stride;
    const Idx stride = Idx(gridDim.x) * (kSelWarps * 32);
    // size is a multiple of 32: every lane of a warp runs the same iterations (the warp-synchronous steps below need it)
    for (Idx k0 = (Idx(blockIdx.x) * kSelWarps + warp) * 32 + lane; k0 < size; k0 += kTopUnroll * stride) {
        typename Cx<T>::type v[kTopUnroll];
#pragma unroll
        for (int u = 0; u < kTopUnroll; ++u)
            if (k0 + u * stride < size) v[u] = st[k0 + u * stride];
#pragma unroll
        for (int u = 0; u < kTopUnroll; ++u) {
            const Idx k = k0 + u * stride;
            if (k < size) {
                const double p = top_prob(v[u]);
                unsigned d = 0;
                const bool ok = top_eligible(p, ta.min_probability) && select_digit(ta.sel, prob_key(p), uint64_t(k) | index_offset, d);
                if (__ballot_sync(0xffffffffu, ok)) {  // one shared-memory add per distinct digit of the warp
                    const unsigned peers = __match_any_sync(0xffffffffu, ok ? d : 0xffffffffu);
                    if (ok && lane == __ffs(peers) - 1) atomicAdd(&h[warp][d], unsigned(__popc(peers)));
                }
            }
        }
    }
    __syncthreads();
    for (int b = threadIdx.x; b < kSelBuckets; b += blockDim.x) {
        uint32_t c = 0;
        for (int w = 0; w < kSelWarps; ++w) c += h[w][b];
        if (c) atomicAdd(&counts[uint64_t(blockIdx.y) * kSelBuckets + b], (unsigned long long)c);
    }
}

__device__ __forceinline__ bool top_taken(const TopCollectArgs& a, const TopCollectArgs* __restrict__ ga, double p, uint64_t kk) {
    if (!top_eligible(p, a.min_probability)) return false;
    const uint64_t key = prob_key(p);
    if (key != a.stop_key) return key < a.stop_key;
    if (a.stop_index == ~0ull) return true;
    uint64_t logical = kk;
    if (a.n_pos) {  // (entries tied with the stop key only)
        logical = 0;
        for (int q = 0; q < a.n_pos; ++q) logical |= ((kk >> ga->pos[q]) & 1ull) << q;
    }
    return logical <= a.stop_index;
}

constexpr int kTopCollectThreads = 256;
constexpr int kTopTile = kTopCollectThreads * kTopUnroll;  // amplitudes per step: kTopUnroll consecutive ones per thread

// grid = (n_cta, entries), block = kTopCollectThreads; CTA c owns the amplitudes [c * seg, (c + 1) * seg) of its entry.
// store == 0: cta_counts[entry][c] = number of entries taken in the segment.  store == 1: each CTA starts at the sum of the
// counts of the CTAs before it and writes its entries in index order (block scan per step): out_index[entry][i] = physical
// index (index_offset | k), out_prob[entry][i] = p, i < capacity.
template <typename T, typename Idx>
__global__ void __launch_bounds__(kTopCollectThreads)
top_collect_kernel(const typename Cx<T>::type* __restrict__ states, uint64_t state_stride, Idx size, Idx seg, uint64_t index_offset,
                   const TopCollectArgs* __restrict__ args, uint32_t* __restrict__ cta_counts, int store, uint64_t capacity,
                   int64_t* __restrict__ out_index, double* __restrict__ out_prob) {
    __shared__ uint32_t s_warp[kTopCollectThreads / 32];
    __shared__ uint64_t s_base;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const TopCollectArgs* ga = args + blockIdx.y;
    const TopCollectArgs a = *ga;
    const auto* st = states + uint64_t(a.entry) * state_stride;
    uint32_t* row_counts = cta_counts + uint64_t(blockIdx.y) * gridDim.x;
    const Idx begin = Idx(blockIdx.x) * seg, end = begin + seg < size ? begin + seg : size;
    uint64_t base = 0;
    if (store) {
        uint64_t before = 0;
        for (unsigned c = threadIdx.x; c < blockIdx.x; c += blockDim.x) before += row_counts[c];
        for (int o = 16; o > 0; o >>= 1) before += __shfl_xor_sync(0xffffffffu, before, o);
        if (threadIdx.x == 0) s_base = 0;
        __syncthreads();
        if (lane == 0 && before) atomicAdd(reinterpret_cast<unsigned long long*>(&s_base), (unsigned long long)before);
        __syncthreads();
        base = s_base;
    }
    uint32_t total = 0;
    for (Idx t = begin; t < end; t += kTopTile) {
        const Idx k0 = t + Idx(threadIdx.x) * kTopUnroll;
        typename Cx<T>::type v[kTopUnroll];
#pragma unroll
        for (int u = 0; u < kTopUnroll; ++u)
            if (k0 + u < end) v[u] = st[k0 + u];
        unsigned flags = 0;
#pragma unroll
        for (int u = 0; u < kTopUnroll; ++u)
            if (k0 + u < end && top_taken(a, ga, top_prob(v[u]), uint64_t(k0 + u) | index_offset)) flags |= 1u << u;
        const uint32_t mine = __popc(flags);
        if (!store) {
            total += mine;
            continue;
        }
        // exclusive prefix of `mine` over the block in thread order
        uint32_t incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t nb = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += nb;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        uint32_t warp_before = 0, step_total = 0;
        for (int w = 0; w < kTopCollectThreads / 32; ++w) {
            const uint32_t c = s_warp[w];
            warp_before += w < warp ? c : 0;
            step_total += c;
        }
        uint64_t at = base + warp_before + incl - mine;
#pragma unroll
        for (int u = 0; u < kTopUnroll; ++u) {
            if ((flags >> u) & 1) {
                if (at < capacity) {
                    out_index[uint64_t(blockIdx.y) * capacity + at] = int64_t(uint64_t(k0 + u) | index_offset);
                    out_prob[uint64_t(blockIdx.y) * capacity + at] = top_prob(v[u]);
                }
                ++at;
            }
        }
        base += step_total;
        __syncthreads();  // s_warp is rewritten by the next step
    }
    if (!store) {
        for (int o = 16; o > 0; o >>= 1) total += __shfl_xor_sync(0xffffffffu, total, o);
        if (threadIdx.x == 0) s_warp[0] = 0;
        __syncthreads();
        if (lane == 0 && total) atomicAdd(&s_warp[0], total);
        __syncthreads();
        if (threadIdx.x == 0) row_counts[blockIdx.x] = s_warp[0];
    }
}

// ---------------------------------------------------------------------------------------------------
// exact marginal probabilities (K11): out[b] = sum of |psi_k|^2 over every k whose measured bits read b, where bit j of b is
// amplitude bit pos[j] (any subset of the index bits, in any order).  One read of the state, no atomics:
//   * a warp reads 32 consecutive amplitudes at a time, so amplitude bits 0..4 are the lane and bits >= 5 the "chunk";
//   * a warp item is (t, s): t fixes the measured chunk bits, s is a slice of the values of the unmeasured chunk bits.  Each lane
//     sums its amplitudes over the slice in ascending order in a register, then an xor-shuffle butterfly over the unmeasured
//     lane bits (ascending) adds up the lanes of one bin; one lane per bin writes part[b][s];
//   * with several slices per t, marginal_reduce_kernel sums part[b][0..S) per bin: threads in slice order, then a fixed tree.
// Every sum's order depends on the bit positions and the state width alone, so two calls give the same bits.  Items are
// independent: the grid only spreads them.  p_k is top_prob's (no FMA contraction), so with every qubit measured out[k] is
// NumPy's re * re + im * im bit for bit.
// ---------------------------------------------------------------------------------------------------
constexpr int kMargMaxBits = 26;    // measured qubits of one call: 2^26 doubles (512 MiB) of output per state
constexpr int kMargWarps = 8;
constexpr int kMargItemBits = 16;   // split a state into about 2^16 warp items: several waves on the device, small partial rows
constexpr int kMargUnroll = 4;      // chunk loads in flight per lane

struct MarginalArgs {
    uint32_t lane_sum;     // amplitude bits 0..4 that are not measured (summed across lanes)
    uint32_t lane_bin[5];  // output bit (1 << j) of amplitude bit b < 5, 0 where not measured
    uint32_t bin_fixed;    // output bits of measured qubits above the state (rank bits of a shard, from index_offset)
    uint32_t fixed_mask;   // the output bits of those qubits: bins with another pattern get no amplitude of this state
    uint32_t v_mask;       // unmeasured chunk bits (amplitude bits >= 5, shifted down by 5)
    int32_t h_bits, v_bits, slice_bits, m;
    int8_t h_pos[32], h_out[32];  // measured chunk bits, ascending, and their output bits
    int8_t v_pos[32];             // unmeasured chunk bits, ascending
};

// grid = (CTAs, states), block = 32 * kMargWarps.  Rows `state_stride` amplitudes apart; out row = 2^(m + slice_bits) doubles,
// [bin][slice] (with slice_bits == 0 the marginal itself).
template <typename T, typename Idx>
__global__ void __launch_bounds__(32 * kMargWarps)
marginal_kernel(const typename Cx<T>::type* __restrict__ states, uint64_t state_stride, MarginalArgs a, double* __restrict__ out) {
    // byte-wise deposit tables of t (measured chunk bits, their output bits) and of the slice start (unmeasured chunk bits)
    __shared__ uint32_t s_hc[4][256], s_hb[4][256], s_vc[4][256];
    for (int e = threadIdx.x; e < 4 * 256; e += blockDim.x) {
        const int byte = e >> 8, x = e & 255;
        uint32_t hc = 0, hb = 0, vc = 0;
        for (int b = 0; b < 8; ++b) {
            const int i = 8 * byte + b;
            if (!((x >> b) & 1)) continue;
            if (i < a.h_bits) hc |= 1u << a.h_pos[i], hb |= 1u << a.h_out[i];
            if (i < a.v_bits) vc |= 1u << a.v_pos[i];
        }
        s_hc[byte][x] = hc, s_hb[byte][x] = hb, s_vc[byte][x] = vc;
    }
    __syncthreads();
    auto deposit = [](const uint32_t (*tab)[256], uint32_t x) { return tab[0][x & 255] | tab[1][(x >> 8) & 255] | tab[2][(x >> 16) & 255] | tab[3][x >> 24]; };
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t lane_bin = a.bin_fixed;
#pragma unroll
    for (int b = 0; b < 5; ++b) lane_bin |= ((lane >> b) & 1) ? a.lane_bin[b] : 0u;
    const auto* st = states + uint64_t(blockIdx.y) * state_stride;
    double* row = out + (uint64_t(blockIdx.y) << (a.m + a.slice_bits));
    const int len_bits = a.v_bits - a.slice_bits;
    const uint64_t len = uint64_t(1) << len_bits, items = uint64_t(1) << (a.h_bits + a.slice_bits);
    const uint32_t slice_mask = (1u << a.slice_bits) - 1u;
    for (uint64_t item = uint64_t(blockIdx.x) * kMargWarps + warp; item < items; item += uint64_t(gridDim.x) * kMargWarps) {  // warp-uniform
        const uint32_t t = uint32_t(item >> a.slice_bits), s = uint32_t(item) & slice_mask;
        const uint32_t hc = deposit(s_hc, t), bin = lane_bin | deposit(s_hb, t);
        uint32_t v = deposit(s_vc, uint32_t(uint64_t(s) << len_bits));
        double acc = 0.0;
        for (uint64_t j = 0; j < len; j += kMargUnroll) {
            typename Cx<T>::type x[kMargUnroll];
#pragma unroll
            for (int u = 0; u < kMargUnroll; ++u) {
                if (j + u < len) {
                    x[u] = st[(Idx(hc | v) << 5) | Idx(lane)];
                    v = ((v | ~a.v_mask) + 1u) & a.v_mask;  // next value of the unmeasured chunk bits
                }
            }
#pragma unroll
            for (int u = 0; u < kMargUnroll; ++u)
                if (j + u < len) acc += top_prob(x[u]);
        }
#pragma unroll
        for (int b = 0; b < 5; ++b)
            if ((a.lane_sum >> b) & 1) acc += __shfl_xor_sync(0xffffffffu, acc, 1 << b);  // a + b == b + a: every lane of a bin agrees
        if ((uint32_t(lane) & a.lane_sum) == 0) row[(uint64_t(bin) << a.slice_bits) | s] = acc;
    }
}

// out[row][b] = sum over s of part[row][b][s]: a group of 2^group_bits threads (32..256, from the slice count) per bin, thread i
// adding s = i, i + G, ... in order, then a fixed xor tree per warp and the group's warps in order.  Bins whose rank-bit pattern
// (fixed_mask) is not this shard's (fixed_value) have no partials and get 0.  grid = (ceil(2^m / bins per block), states), block = 256.
__global__ void __launch_bounds__(256)
marginal_reduce_kernel(const double* __restrict__ part, int m, int slice_bits, int group_bits, uint32_t fixed_mask, uint32_t fixed_value,
                       double* __restrict__ out) {
    __shared__ double s_w[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = threadIdx.x >> group_bits, i = threadIdx.x & ((1 << group_bits) - 1);
    const uint64_t bin = (uint64_t(blockIdx.x) << (8 - group_bits)) + g;
    const bool live = bin < (uint64_t(1) << m) && (uint32_t(bin) & fixed_mask) == fixed_value;
    double acc = 0.0;
    if (live) {
        const double* p = part + (uint64_t(blockIdx.y) << (m + slice_bits)) + (bin << slice_bits);
        for (uint64_t s = i; s < (uint64_t(1) << slice_bits); s += (1u << group_bits)) acc += p[s];
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (group_bits > 5) {
        if (lane == 0) s_w[warp] = acc;
        __syncthreads();
        if (i == 0) {
            acc = 0.0;
            for (int w = 0; w < (1 << (group_bits - 5)); ++w) acc += s_w[(g << (group_bits - 5)) + w];
        }
    }
    if (i == 0 && bin < (uint64_t(1) << m)) out[(uint64_t(blockIdx.y) << m) + bin] = acc;
}

// ---------------------------------------------------------------------------------------------------
// global <-> local qubit swap of a sharded state, fused with its all-to-all: every rank streams its shard ONCE and stores
// each amplitude straight into the peer that owns it afterwards (peer-mapped buffers, NVLink 5 / NVSwitch), already at its
// final position -- no pack pass, no staging buffer, no unpack pass.
//   element i of rank r (local bits lp = d) -> rank d, element i with the lp bits replaced by r
// ---------------------------------------------------------------------------------------------------
constexpr int kMaxSwapRanks = 16;
struct SwapArgs {
    void* peer[kMaxSwapRanks];  // destination buffer of every rank (peer[rank] = own spare buffer)
    int32_t lp[4];              // local bit positions exchanged with rank bits 0..g-1, ascending
    int32_t g, rank;
    int32_t run_bits;           // log2 of the run length (kSwapRunBits, less for tiny shards)
};

// Work order: the shard is cut into runs of 2^kSwapRunBits amplitudes; consecutive runs go to different destination ranks
// (run number XOR own rank), so at any moment every GPU stores to all of its peers and no two GPUs gang up on one receiver --
// a linear walk would have all ranks write into the same peer at the same time (measured: 277 GB/s instead of ~650).
constexpr int kSwapRunBits = 10;

template <typename C>
__global__ void __launch_bounds__(256)
swap_p2p_kernel(const C* __restrict__ src, SwapArgs args, uint64_t size) {
    uint64_t lpmask = 0, rbits = 0;
    for (int j = 0; j < args.g; ++j) {
        lpmask |= 1ull << args.lp[j];
        rbits |= uint64_t((args.rank >> j) & 1) << args.lp[j];
    }
    const int g = args.g;
    const int rb = args.run_bits;
    const uint64_t run_mask = (1ull << rb) - 1ull, dmask = (1ull << g) - 1ull;
    // element number t -> (destination d, index j among the amplitudes bound for d) -> shard index i
    auto locate = [&](uint64_t t, int& d) -> uint64_t {
        d = int((t >> rb) & dmask) ^ args.rank;
        uint64_t i = ((t >> (rb + g)) << rb) | (t & run_mask);
        for (int j = 0; j < g; ++j) {  // lp ascending: open a gap at each exchanged position and drop d's bit in
            const int p = args.lp[j];
            i = ((i >> p) << (p + 1)) | (i & ((1ull << p) - 1ull)) | (uint64_t((d >> j) & 1) << p);
        }
        return i;
    };
    const uint64_t stride = uint64_t(gridDim.x) * blockDim.x;
    constexpr int kUnroll = 4;
    for (uint64_t t0 = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; t0 < size; t0 += stride * kUnroll) {
        C v[kUnroll];
        uint64_t at[kUnroll];
        int dst[kUnroll];
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
            const uint64_t t = t0 + u * stride;
            if (t < size) {
                at[u] = locate(t, dst[u]);
                v[u] = src[at[u]];
            }
        }
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
            const uint64_t t = t0 + u * stride;
            if (t < size) static_cast<C*>(args.peer[dst[u]])[(at[u] & ~lpmask) | rbits] = v[u];
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// The same exchange in place, one buffer per rank.  Swapping the g rank bits with the local bits lp is an involution: element i
// of rank r whose lp bits read d != r trades places with element i' = (i & ~lpmask) | rbits(r) of rank d; elements with d == r
// stay.  One thread swaps a pair (loads both, stores both crosswise); no other thread on any GPU touches those two addresses.
// Pair ownership: p0 = the highest local bit not in lp is the same in i and i'; rank r handles the pair iff that bit is (r > d),
// so exactly one of the two ranks does (a high owner bit keeps the accesses of neighbouring items contiguous).  Each rank moves half of its cross elements toward every peer: half of the bytes cross
// NVLink as remote loads, half as remote stores, the same bytes per GPU and direction as swap_p2p_kernel.
// ---------------------------------------------------------------------------------------------------
struct SwapInplaceArgs {
    void* state[kMaxSwapRanks];  // every rank's state buffer, peer-mapped (state[rank] = own)
    uint64_t lpmask, rbits;      // exchanged local bits; this rank's bits dropped in at them
    int32_t ins_pos[5];          // the g + 1 inserted bit positions (lp and p0), ascending
    int32_t ins_src[5];          // bit of (d | owner << g) that goes to ins_pos[s]: j < g = bit j of d, g = the owner bit
    int32_t g, rank;
    int32_t run_bits;            // log2 of the run length, <= n_local - g - 1
};

// Remote loads have to cover the NVLink round trip with bytes in flight: twice the pairs per thread of swap_p2p_kernel's elements.
constexpr int kInplaceUnroll = 8;

// Work order (as in swap_p2p_kernel): items t < (W-1) 2^(n_local-g-1), run u = t >> run_bits goes to peer d = rank ^ (1 + u % (W-1)),
// so at any item number the ranks target pairwise different peers and each rank rotates over all of its peers.  Within a peer
// the pair number is ((u / (W-1)) << run_bits) | (t & run_mask), expanded to i by dropping in d's bits at lp and the owner bit at p0.
template <typename C>
__global__ void __launch_bounds__(256)
swap_inplace_p2p_kernel(SwapInplaceArgs args, uint64_t items) {
    const int g = args.g, rank = args.rank, rb = args.run_bits;
    const uint32_t peers = (1u << g) - 1u;
    const uint64_t run_mask = (1ull << rb) - 1ull;
    C* __restrict__ own = static_cast<C*>(args.state[rank]);
    auto locate = [&](uint64_t t, int& d) -> uint64_t {
        const uint32_t u = uint32_t(t >> rb);  // < (W-1) 2^(n_local-g-1-run_bits) < 2^32 for n_local <= 36
        const uint32_t k = 1u + u % peers;
        d = rank ^ int(k);
        const uint32_t bits = uint32_t(d) | (uint32_t(rank > d) << g);
        uint64_t i = (uint64_t(u / peers) << rb) | (t & run_mask);
        for (int s = 0; s <= g; ++s) {  // ascending: open a gap at each inserted position and drop its bit in
            const int p = args.ins_pos[s];
            i = ((i >> p) << (p + 1)) | (i & ((1ull << p) - 1ull)) | (uint64_t((bits >> args.ins_src[s]) & 1u) << p);
        }
        return i;
    };
    const uint64_t stride = uint64_t(gridDim.x) * blockDim.x;
    for (uint64_t t0 = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; t0 < items; t0 += stride * kInplaceUnroll) {
        C a[kInplaceUnroll], b[kInplaceUnroll];
        C* there[kInplaceUnroll];
        uint64_t at[kInplaceUnroll];
#pragma unroll
        for (int u = 0; u < kInplaceUnroll; ++u) {
            const uint64_t t = t0 + u * stride;
            if (t < items) {
                int d;
                at[u] = locate(t, d);
                there[u] = static_cast<C*>(args.state[d]) + ((at[u] & ~args.lpmask) | args.rbits);
                a[u] = __ldcg(own + at[u]);
                b[u] = __ldcg(there[u]);
            }
        }
#pragma unroll
        for (int u = 0; u < kInplaceUnroll; ++u) {
            const uint64_t t = t0 + u * stride;
            if (t < items) {
                own[at[u]] = b[u];
                *there[u] = a[u];
            }
        }
    }
}

template <typename T>
__global__ void to_c128_kernel(const typename Cx<T>::type* __restrict__ src, double2* __restrict__ dst, uint64_t size) {
    for (uint64_t k = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; k < size; k += uint64_t(gridDim.x) * blockDim.x) {
        const auto a = src[k];
        dst[k] = make_double2(double(a.x), double(a.y));
    }
}

}  // namespace qb
