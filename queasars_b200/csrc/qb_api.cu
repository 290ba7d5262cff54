// C-ABI implementation (include/queasars_b200.h): contexts, plans, Hamiltonians, batched evaluation.
// No CPU fallback: every compute entry point needs a CUDA device and fails with QB_ERR_CUDA otherwise.
#include <algorithm>
#include <cmath>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <tuple>
#include <functional>
#include <memory>
#include <mutex>
#include <numeric>
#include <string>
#include <thread>
#include <vector>

#include <cub/device/device_radix_sort.cuh>

#include "qb_kernels.cuh"

namespace {

thread_local std::string g_last_error;

int fail(int code, const std::string& msg) {
    g_last_error = msg;
    return code;
}

#define QB_CUDA(call)                                                                                      \
    do {                                                                                                   \
        cudaError_t qb_e_ = (call);                                                                        \
        if (qb_e_ != cudaSuccess)                                                                          \
            return fail(QB_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(qb_e_));               \
    } while (0)

#define QB_TRY(call)                 \
    do {                             \
        int qb_r_ = (call);          \
        if (qb_r_ != QB_OK) return qb_r_; \
    } while (0)

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return QB_OK;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail(QB_ERR_MEMORY, "cudaMalloc of " + std::to_string(bytes) + " bytes failed: " + cudaGetErrorString(e));
        }
        cap = bytes;
        return QB_OK;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct HostBuf {  // pinned staging
    void* p = nullptr;
    size_t cap = 0;
    bool mapped = false;  // small buffers kernels read / write directly (device alias: device_ptr())
    int reserve(size_t bytes) {
        if (bytes <= cap) return QB_OK;
        if (p) cudaFreeHost(p);  // callers synchronise on the buffer's event before growing it
        p = nullptr;
        cap = 0;
        size_t want = std::max<size_t>(bytes, mapped ? 4096 : (1 << 16));
        cudaError_t e = cudaHostAlloc(&p, want, mapped ? (cudaHostAllocMapped | cudaHostAllocPortable) : cudaHostAllocDefault);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail(QB_ERR_MEMORY, std::string("cudaHostAlloc failed: ") + cudaGetErrorString(e));
        }
        cap = want;
        return QB_OK;
    }
    void* device_ptr() const {
        void* d = nullptr;
        if (!p || cudaHostGetDevicePointer(&d, p, 0) != cudaSuccess) {
            cudaGetLastError();
            return nullptr;
        }
        return d;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
};

struct Plan {
    int n_qubits = 0, n_eff = 0, dtype = 0, tile_bits = QB_TILE_BITS, reg_bits = 4, n_params = 0, n_ops = 0, n_sweeps = 0, n_pass_ops = 0;
    DevBuf sweeps, passes, pass_ops, angles, init_ops;
    bool has_init = false;
    int64_t prefix_id = 0;     // parameter-free plan whose result this plan starts from (0: none)
    DevBuf prefix_state;       // cached result of the prefix plan
    bool prefix_ready = false;
    ~Plan() { sweeps.release(), passes.release(), pass_ops.release(), angles.release(), init_ops.release(), prefix_state.release(); }
};

struct Group {
    uint64_t xmask = 0;
    int n_terms = 0;
    DevBuf z, wr, wi;
};

struct Ham {
    int n_qubits = 0;
    int n_diag = 0;       // number of z-only terms (device arrays diag_z / diag_c, real coefficients)
    bool diagonal = true;  // no x-mask anywhere
    DevBuf diag_z, diag_c;
    std::vector<std::unique_ptr<Group>> groups;  // x == 0 group first (if any), complex weights
    DevBuf table;
    int table_n_eff = 0;
    // tile-fused evaluation of the non-diagonal groups (expect_tile_kernel); groups that do not fit a tile stay generic
    std::vector<qb::ExpTileSweep> tile_sweeps;
    std::vector<std::vector<int>> tile_sweep_groups;  // indices into `groups` evaluated by each tile sweep
    std::vector<int> generic_groups;  // indices into `groups`
    DevBuf tile_groups, tile_z, tile_wr, tile_wi;
    int tile_n_eff = 0;
    // data of the exact CVaR (qb_evaluate_cvar), built on first use: E(k) in basis order (every alpha), and for alpha < 1 the
    // stable ascending (E, k) order as sorted position -> basis index with E at each sorted position
    DevBuf cvar_energy, cvar_perm, cvar_sorted;
    int cvar_energy_n_eff = 0, cvar_order_n_eff = 0;
    ~Ham() {
        cvar_energy.release(), cvar_perm.release(), cvar_sorted.release();
        tile_groups.release(), tile_z.release(), tile_wr.release(), tile_wi.release();
        diag_z.release(), diag_c.release(), table.release();
        for (auto& g : groups) g->z.release(), g->wr.release(), g->wi.release();
    }
};

// A set of observables evaluated together (qb_evaluate_observables): the union of their distinct Pauli strings, grouped by
// x mask and planned into tile sweeps like a Hamiltonian's groups, plus the CSR rows that combine string values into observables.
struct Obs {
    int n_qubits = 0, n_obs = 0, n_terms = 0, n_eff = 0;
    std::vector<qb::ExpTileSweep> tile_sweeps;
    std::vector<std::pair<int, int>> sweep_terms;  // device term range of every tile sweep
    std::vector<qb::TermGroup> generic;            // groups whose x mask does not fit a tile (term ranges on the device)
    DevBuf groups, z, im, sign, row_begin, cols, coeff;
    ~Obs() { groups.release(), z.release(), im.release(), sign.release(), row_begin.release(), cols.release(), coeff.release(); }
};

// A set of circuit evaluations resident on the device.
struct DeviceBatch {
    int batch = 0, n_eff = 0, n_qubits = 0, dtype = 0, tile_bits = QB_TILE_BITS, reg_bits = 4, max_sweeps = 0;
    std::vector<int> order;   // sorted position -> caller index (descending sweep count)
    std::vector<int> active;  // active[s] = number of entries with more than s sweeps
    std::vector<qb::BatchEntry> h_entries;
    std::vector<int64_t> param_begin;  // per caller index, offset into the params buffer
    int64_t total_params = 0, total_ops = 0;
    const Ham* ham = nullptr;
    int64_t ham_id = 0;  // resident batches: the Hamiltonian is looked up again by id whenever the batch is re-assembled
    // what the buffers were last assembled for: an identical request (same plans, Hamiltonian, start) re-uses them as they are
    std::vector<int64_t> built_ids;
    uint64_t built_epoch = 0, built_offset = 0;
    int built_init_zero = -1;
    bool fuse_expect = false;
    bool skip_final_store = false;  // fused diagonal <H> is the whole result: the last sweep does not write the state back
    size_t n_tiles = 0, partial_stride = 0;
    int tiles_log2 = 0;  // every sweep CTA walks 2^tiles_log2 consecutive tiles (and writes ONE fused-expectation partial)
    int64_t n_state_sweeps = 0, launches_per_run = 0;
    DevBuf entries, params, matrices, partials, out, states;
    bool owns_states = true;
    // low-latency single-circuit path (cached CUDA graph): bind_kernel reads the parameters from, and the last reduction writes
    // the value to, mapped pinned host memory (no copy nodes); the kernels of the chain are launched programmatically dependent
    const double* params_mapped = nullptr;
    double* out_mapped = nullptr;
    bool pdl = false;
    ~DeviceBatch() {
        entries.release(), params.release(), matrices.release(), partials.release(), out.release();
        if (owns_states) states.release();
    }
};

// One host thread per context for qb_evaluate_expectation_multi: a caller that drives several GPUs hands every context its share
// and all of them build, launch and wait concurrently -- outside the interpreter lock of a Python caller, which is what makes a
// single process able to keep several GPUs busy with small shares.
struct Worker {
    std::thread thread;
    std::mutex m;
    std::condition_variable cv;
    std::function<int()> task;
    bool has_task = false, done = false, stop = false;
    int rc = QB_OK;
    std::string error;

    void loop() {
        std::unique_lock<std::mutex> lock(m);
        for (;;) {
            cv.wait(lock, [&] { return has_task || stop; });
            if (stop) return;
            std::function<int()> fn = std::move(task);
            has_task = false;
            lock.unlock();
            const int r = fn();
            std::string msg = r == QB_OK ? std::string() : g_last_error;  // (thread-local: this thread's)
            lock.lock();
            rc = r, error = std::move(msg), done = true;
            cv.notify_all();
        }
    }
    void post(std::function<int()> fn) {
        std::lock_guard<std::mutex> lock(m);
        task = std::move(fn), has_task = true, done = false;
        cv.notify_all();
    }
    int wait(std::string& msg) {
        std::unique_lock<std::mutex> lock(m);
        cv.wait(lock, [&] { return done; });
        msg = error;
        return rc;
    }
    ~Worker() {
        {
            std::lock_guard<std::mutex> lock(m);
            stop = true;
            cv.notify_all();
        }
        if (thread.joinable()) thread.join();
    }
};

// One (plan, Hamiltonian) evaluation captured as a CUDA graph: parameter upload from a fixed pinned buffer, bind, sweeps,
// expectation, result download into a fixed pinned buffer.  Replayed by the single-circuit calls of an optimizer loop
// (mutation.py:63-75 re-submits ONE circuit with new parameter values), where launch latency, not the GPU, sets the pace.
struct SingleGraph {
    DeviceBatch batch;
    HostBuf pin_params, pin_out;
    cudaGraphExec_t exec = nullptr;
    uint64_t last_use = 0;
    size_t state_bytes = 0;
    ~SingleGraph() {
        if (exec) cudaGraphExecDestroy(exec);
        pin_params.release(), pin_out.release();
    }
};

}  // namespace

struct qb_context {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool owns_stream = false;
    int sm_count = 148;
    uint64_t workspace_limit = 0;
    uint64_t default_workspace = uint64_t(8) << 30;  // 80 % of the memory free at creation (cudaMemGetInfo is slow: ask once)
    int64_t launches = 0;
    int64_t next_id = 1;
    uint64_t epoch = 1;  // bumped whenever a plan or Hamiltonian is destroyed (invalidates assembled batches that may point into it)
    int l2_prefetch = 1;    // QB_L2_PREFETCH=0 switches the next-tile L2 prefetch of the sweep kernel off
    int sweep_group = 0;    // QB_SWEEP_GROUP: circuits per group (0: batch / sweep_streams)
    int sweep_streams = 2;  // QB_SWEEP_STREAMS: groups of circuits whose sweep launches run on separate streams (tail overlap)
    cudaStream_t aux_streams[8] = {};
    cudaEvent_t fork_event = nullptr, join_events[8] = {};
    bool force_idx64 = false;  // qb_context_set_index_width(64): run the 64-bit-index sweep kernels at any size (tests)
    int tiles_log2 = -1;  // tiles per sweep CTA (log2); -1 = 8 tiles, fewer while a launch would not fill two waves of CTAs; QB_TILES_LOG2 overrides
    std::mutex mu;
    std::map<int64_t, std::unique_ptr<Plan>> plans;
    std::map<int64_t, std::unique_ptr<Ham>> hams;
    std::map<int64_t, std::unique_ptr<Obs>> observables;
    std::map<int64_t, std::unique_ptr<DeviceBatch>> batches;
    HostBuf pin_in, pin_out, pin_entries;
    cudaEvent_t pin_entries_done = nullptr;
    cudaEvent_t pin_in_done = nullptr;  // last H2D copy out of pin_in
    DevBuf scratch;                     // uniforms / indices / chunk sums / single-state partials
    DeviceBatch oneshot;                // buffers reused by the one-shot entry points (no per-call cudaMalloc)
    // pipelined submission (qb_evaluate_expectation_submit / _collect): results of queued chunks land here
    struct PendingChunk {
        size_t offset;           // first result slot in pin_res
        std::vector<int> order;  // sorted device position -> index inside the chunk
    };
    HostBuf pin_res;
    std::vector<PendingChunk> pending;
    size_t pending_results = 0;
    // single-evaluation graphs (qb_evaluate_expectation with batch == 1), least recently used evicted first
    bool use_graphs = true;  // QB_GRAPHS=0 disables
    bool zero_copy = true;   // QB_ZERO_COPY=0: single-circuit graphs copy parameters / value with memcpy nodes instead of mapped pinned memory
    int pdl = 1;             // QB_PDL: 0 off, 1 programmatic dependent launches inside the single-circuit graphs, 2 for every sweep chain
    std::map<std::tuple<int64_t, int64_t, int>, std::unique_ptr<SingleGraph>> single_graphs;  // (plan, Hamiltonian, copies)
    size_t single_graph_bytes = 0;
    uint64_t use_clock = 0;
    std::unique_ptr<Worker> worker;  // created by the first qb_evaluate_expectation_multi that includes this context
    std::mutex worker_mu;
};

namespace {

size_t amp_bytes(int dtype) { return dtype == QB_C128 ? 16 : 8; }

size_t workspace_limit_of(const qb_context* ctx) { return ctx->workspace_limit ? ctx->workspace_limit : ctx->default_workspace; }

// f(double()) for complex128 amplitudes, f(float()) for every other dtype code: `using T = decltype(t);` picks the kernel instance
template <typename F> int with_dtype(int dtype, F&& f) { return dtype == QB_C128 ? f(double()) : f(float()); }

// rows of `row_bytes` between sorted device position pos and caller index order[pos]: scatter_rows puts device rows in caller
// order, gather_rows caller rows in device order
void scatter_rows(void* caller, const void* device, const std::vector<int>& order, size_t row_bytes) {
    for (size_t pos = 0; pos < order.size(); ++pos)
        std::memcpy(static_cast<char*>(caller) + size_t(order[pos]) * row_bytes, static_cast<const char*>(device) + pos * row_bytes, row_bytes);
}
void gather_rows(void* device, const void* caller, const std::vector<int>& order, size_t row_bytes) {
    for (size_t pos = 0; pos < order.size(); ++pos)
        std::memcpy(static_cast<char*>(device) + pos * row_bytes, static_cast<const char*>(caller) + size_t(order[pos]) * row_bytes, row_bytes);
}

// terms of one x-mask group staged in shared memory (24 B each, inside the default 48 KB); longer lists are read from global memory
constexpr int kMaxStagedTerms = 2000;
// diagonal terms per diag_table_kernel launch (16 B each in shared memory); longer lists build the table in several launches
constexpr int kTableTermChunk = 3000;

// Every entry point works on its context's device and gives the calling thread its previous current device back on return: a host
// program that drives several engines from one thread, or shares the thread with torch (bench.py, sharded.py), must not find its
// current device changed behind its back (torch then allocates, and runs NCCL collectives, on the wrong GPU).
struct DeviceScope {
    int prev = -1, dev;
    cudaError_t err;
    explicit DeviceScope(int device) : dev(device) {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != dev) err = cudaSetDevice(dev);
    }
    ~DeviceScope() {
        if (prev >= 0 && prev != dev) cudaSetDevice(prev);
    }
    DeviceScope(const DeviceScope&) = delete;
    DeviceScope& operator=(const DeviceScope&) = delete;
};

#define QB_ON_DEVICE(ctx)                                                                                   \
    DeviceScope qb_scope_((ctx)->device);                                                                   \
    if (qb_scope_.err != cudaSuccess) return fail(QB_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(qb_scope_.err))

template <typename K> int configure_kernel(K kernel, size_t smem) {
    QB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    // QB_SMEM_CARVEOUT = 0..100: preferred shared-memory share of the SM's unified L1 / shared storage (default: the driver's choice)
    if (const char* e = std::getenv("QB_SMEM_CARVEOUT")) QB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, std::atoi(e)));
    return QB_OK;
}

int check_launch(qb_context* ctx, const char* what) {
    ctx->launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(QB_ERR_CUDA, std::string(what) + " launch failed: " + cudaGetErrorString(e));
    return QB_OK;
}

// Kernel launch, optionally programmatically dependent on the kernel before it in the stream (see pdl_wait() in qb_kernels.cuh).
template <typename... KArgs, typename... Args>
void launch_kernel(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, bool pdl, Args... args) {
    if (!pdl) {
        kernel<<<grid, block, smem, stream>>>(KArgs(args)...);
        return;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid, cfg.blockDim = block, cfg.dynamicSmemBytes = smem, cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr, cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);  // errors surface in check_launch
}

int upload(qb_context* ctx, DevBuf& dst, const void* src, size_t bytes) {
    QB_TRY(dst.reserve(std::max<size_t>(bytes, 16)));
    if (bytes) QB_CUDA(cudaMemcpyAsync(dst.p, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return QB_OK;
}

Plan* find_plan(qb_context* ctx, int64_t id) {
    auto it = ctx->plans.find(id);
    return it == ctx->plans.end() ? nullptr : it->second.get();
}

Ham* find_ham(qb_context* ctx, int64_t id) {
    auto it = ctx->hams.find(id);
    return it == ctx->hams.end() ? nullptr : it->second.get();
}

int build_batch(qb_context* ctx, DeviceBatch& b, int batch, const int64_t* plan_ids, const Ham* ham, void* external_state,
                int init_zero, uint64_t index_offset);
int launch_circuits(qb_context* ctx, DeviceBatch& b, cudaEvent_t* events);

// Compute (once) the state a prefixed plan starts from: run the parameter-free prefix plan into a buffer owned by the plan.
int ensure_prefix_state(qb_context* ctx, Plan* pl) {
    if (!pl->prefix_id || pl->prefix_ready) return QB_OK;
    Plan* pre = find_plan(ctx, pl->prefix_id);
    if (!pre) return fail(QB_ERR_NOT_FOUND, "prefix plan " + std::to_string(pl->prefix_id) + " no longer exists");
    if (pre->n_eff != pl->n_eff || pre->dtype != pl->dtype || pre->n_params != 0 || pre->prefix_id)
        return fail(QB_ERR_INVALID, "prefix plan must be parameter-free, un-prefixed and of the same shape");
    const size_t state_bytes = (size_t(1) << pl->n_eff) * amp_bytes(pl->dtype);
    QB_TRY(pl->prefix_state.reserve(state_bytes));
    DeviceBatch tmp;
    QB_TRY(build_batch(ctx, tmp, 1, &pl->prefix_id, nullptr, pl->prefix_state.p, 1, 0));
    QB_TRY(launch_circuits(ctx, tmp, nullptr));
    QB_CUDA(cudaStreamSynchronize(ctx->stream));  // tmp's small device buffers are released when it goes out of scope
    pl->prefix_ready = true;
    return QB_OK;
}

// ---- batch assembly -------------------------------------------------------------------------------
int build_batch(qb_context* ctx, DeviceBatch& b, int batch, const int64_t* plan_ids, const Ham* ham, void* external_state,
                int init_zero, uint64_t index_offset) {
    if (batch <= 0) return fail(QB_ERR_INVALID, "batch must be positive");
    // The same list as last time (an optimizer loop, one generation evaluated again): entries, buffers and launch shape are
    // still valid on the device -- nothing to assemble or upload.  `epoch` moves whenever a plan or Hamiltonian is destroyed.
    if (!external_state && b.owns_states && b.batch == batch && b.ham == ham && b.built_epoch == ctx->epoch && b.built_init_zero == init_zero &&
        b.built_offset == index_offset && b.built_ids.size() == size_t(batch) && std::memcmp(b.built_ids.data(), plan_ids, sizeof(int64_t) * size_t(batch)) == 0)
        return QB_OK;
    b.built_ids.clear();
    std::vector<Plan*> plans(batch);
    for (int i = 0; i < batch; ++i) {
        plans[i] = find_plan(ctx, plan_ids[i]);
        if (!plans[i]) return fail(QB_ERR_NOT_FOUND, "unknown plan id " + std::to_string(plan_ids[i]));
        if (plans[i]->n_eff != plans[0]->n_eff || plans[i]->dtype != plans[0]->dtype || plans[i]->n_qubits != plans[0]->n_qubits ||
            plans[i]->reg_bits != plans[0]->reg_bits || plans[i]->tile_bits != plans[0]->tile_bits)
            return fail(QB_ERR_INVALID, "all plans of one batch must share qubit count, dtype and tile / register-bit counts");
    }
    for (int i = 0; i < batch; ++i)
        if (plans[i]->prefix_id && (external_state || !init_zero))
            return fail(QB_ERR_INVALID, "a plan with a cached prefix state cannot be applied to an external state");
    for (int i = 0; i < batch; ++i) QB_TRY(ensure_prefix_state(ctx, plans[i]));
    if (!init_zero)
        for (int i = 0; i < batch; ++i)
            if (plans[i]->has_init) return fail(QB_ERR_INVALID, "plan was compiled for a |0...0> start (product-state prefix) but is applied to an existing state");
    b.batch = batch;
    b.n_eff = plans[0]->n_eff;
    b.n_qubits = plans[0]->n_qubits;
    b.dtype = plans[0]->dtype;
    b.reg_bits = plans[0]->reg_bits;
    b.tile_bits = plans[0]->tile_bits;
    b.ham = ham;
    if (ham && ham->n_qubits != b.n_qubits)
        return fail(QB_ERR_INVALID, "Hamiltonian acts on " + std::to_string(ham->n_qubits) + " qubits, circuits on " + std::to_string(b.n_qubits));
    b.fuse_expect = ham && ham->table.p && ham->table_n_eff == b.n_eff && index_offset == 0;  // diagonal part in the last sweep
    b.skip_final_store = b.fuse_expect && ham->diagonal && !external_state;
    b.n_tiles = size_t(1) << (b.n_eff - b.tile_bits);
    // 8 tiles per CTA: the staging of the sweep program (pass records, matrices, slot tables: ~8 % of the warp time at 4 tiles) is
    // paid once per 8 tiles; with the sweep launches overlapping as stream groups the longer CTAs no longer cost a tail
    // (measured on the bench workload: 1 / 2 / 4 / 8 / 16 tiles per CTA -> 25.3 / 28.9 / 31.3 / 32.2 / 30.5 k evals/s)
    b.tiles_log2 = std::min(ctx->tiles_log2 >= 0 ? ctx->tiles_log2 : 3, b.n_eff - b.tile_bits);
    if (ctx->tiles_log2 < 0) {  // small batches: rather more CTAs than amortised staging -- keep at least two waves of them
        const size_t slots = size_t(ctx->sm_count) * (b.tile_bits <= 11 ? 4 : 2);
        while (b.tiles_log2 > 0 && ((b.n_tiles * size_t(batch)) >> b.tiles_log2) < 2 * slots) --b.tiles_log2;
    }
    b.partial_stride = std::max<size_t>(size_t(1) << (b.n_eff - std::min(b.n_eff, qb::kExpTileBits)), std::max<size_t>(b.n_tiles, 1024));

    b.order.resize(batch);
    std::iota(b.order.begin(), b.order.end(), 0);
    std::stable_sort(b.order.begin(), b.order.end(), [&](int x, int y) { return plans[x]->n_sweeps > plans[y]->n_sweeps; });
    b.max_sweeps = plans[b.order[0]]->n_sweeps;
    b.active.assign(b.max_sweeps, 0);
    b.param_begin.assign(batch + 1, 0);
    std::vector<int64_t> op_begin(batch + 1, 0);
    b.n_state_sweeps = 0;
    for (int i = 0; i < batch; ++i) {
        b.param_begin[i + 1] = b.param_begin[i] + plans[i]->n_params;
        op_begin[i + 1] = op_begin[i] + plans[i]->n_ops + plans[i]->n_pass_ops + (plans[i]->n_eff + 1) / 2;  // + 4 doubles per qubit
        for (int s = 0; s < plans[i]->n_sweeps; ++s) b.active[s]++;
        b.n_state_sweeps += plans[i]->n_sweeps;
    }
    b.total_params = b.param_begin[batch];
    b.total_ops = op_begin[batch];

    const size_t state_bytes = (size_t(1) << b.n_eff) * amp_bytes(b.dtype);
    if (external_state) {
        if (batch != 1) return fail(QB_ERR_INVALID, "external state needs batch == 1");
        b.owns_states = false;
        b.states.p = external_state;
    } else {
        const size_t need = state_bytes * size_t(batch);
        if (ctx->workspace_limit && need > ctx->workspace_limit)
            return fail(QB_ERR_MEMORY, "batch needs " + std::to_string(need) + " bytes of statevector workspace, limit is " +
                                           std::to_string(ctx->workspace_limit));
        QB_TRY(b.states.reserve(need));
    }
    QB_TRY(b.params.reserve(std::max<size_t>(sizeof(double) * size_t(b.total_params), 16)));
    QB_TRY(b.matrices.reserve(std::max<size_t>(sizeof(double) * 8 * size_t(b.total_ops), 64)));
    QB_TRY(b.partials.reserve(sizeof(double) * b.partial_stride * size_t(batch)));
    QB_TRY(b.out.reserve(sizeof(double) * size_t(batch)));

    b.h_entries.resize(batch);
    for (int pos = 0; pos < batch; ++pos) {
        const int i = b.order[pos];
        const Plan* pl = plans[i];
        qb::BatchEntry& en = b.h_entries[pos];
        en.sweeps = pl->sweeps.as<qb_sweep>();
        en.passes = pl->passes.as<qb_pass>();
        en.pass_ops = pl->pass_ops.as<qb_pass_op>();
        en.angles = pl->angles.as<qb_op_angles>();
        en.init_ops = pl->has_init ? pl->init_ops.as<int32_t>() : nullptr;
        en.params = (b.params_mapped ? b.params_mapped : b.params.as<double>()) + b.param_begin[i];
        en.matrices = b.matrices.as<double>() + 8 * op_begin[i];
        en.state = static_cast<unsigned char*>(b.states.p) + state_bytes * size_t(pos);
        en.src_state = pl->prefix_id ? pl->prefix_state.p : nullptr;
        en.diag_table = b.fuse_expect ? ham->table.as<double>() : nullptr;
        en.partials = b.partials.as<double>() + b.partial_stride * size_t(pos);
        en.n_sweeps = pl->n_sweeps;
        en.n_ops = pl->n_ops;
        en.n_pass_ops = pl->n_pass_ops;
        en.n_init = pl->n_eff;
        en.n_params = pl->n_params;
        en.init_zero = pl->prefix_id ? 0 : init_zero;
        en.index_offset = index_offset;
    }
    {   // entries go through the pinned staging buffer so the copy is truly asynchronous
        const size_t bytes = sizeof(qb::BatchEntry) * size_t(batch);
        QB_TRY(b.entries.reserve(bytes));
        QB_CUDA(cudaEventSynchronize(ctx->pin_entries_done));  // before a possible re-allocation: a copy out of it may be queued
        QB_TRY(ctx->pin_entries.reserve(bytes));
        std::memcpy(ctx->pin_entries.p, b.h_entries.data(), bytes);
        QB_CUDA(cudaMemcpyAsync(b.entries.p, ctx->pin_entries.p, bytes, cudaMemcpyHostToDevice, ctx->stream));
        QB_CUDA(cudaEventRecord(ctx->pin_entries_done, ctx->stream));
    }
    if (!external_state) {
        b.built_ids.assign(plan_ids, plan_ids + batch);
        b.built_epoch = ctx->epoch, b.built_offset = index_offset, b.built_init_zero = init_zero;
    }
    return QB_OK;
}

int batch_upload_params(qb_context* ctx, DeviceBatch& b, const double* params, const int64_t* param_offsets) {
    if (b.total_params == 0) return QB_OK;
    QB_CUDA(cudaEventSynchronize(ctx->pin_in_done));
    QB_TRY(ctx->pin_in.reserve(sizeof(double) * size_t(b.total_params)));
    double* stage = static_cast<double*>(ctx->pin_in.p);
    for (int i = 0; i < b.batch; ++i) {
        const int64_t n = b.param_begin[i + 1] - b.param_begin[i];
        if (param_offsets[i + 1] - param_offsets[i] != n)
            return fail(QB_ERR_INVALID, "entry " + std::to_string(i) + ": got " + std::to_string(param_offsets[i + 1] - param_offsets[i]) +
                                            " parameter values, circuit has " + std::to_string(n) + " parameters");
        std::memcpy(stage + b.param_begin[i], params + param_offsets[i], sizeof(double) * size_t(n));
    }
    QB_CUDA(cudaMemcpyAsync(b.params.p, stage, sizeof(double) * size_t(b.total_params), cudaMemcpyHostToDevice, ctx->stream));
    QB_CUDA(cudaEventRecord(ctx->pin_in_done, ctx->stream));
    return QB_OK;
}

// Sweep launches of one batch.  A sweep launch is a full drain point: the next sweep of ANY circuit waits for the slowest CTA of
// this one.  With `sweep_streams` > 1 the (sorted) batch is cut into that many contiguous groups of circuits, each group runs its
// own sweeps back to back on its own stream, so the tail of one group's launch overlaps the next launch of another group
// (circuits are independent: no ordering between groups is needed).  Event-timed runs keep the single stream.
template <typename T, int R, int K, typename Idx> int launch_sweeps_t(qb_context* ctx, DeviceBatch& b, cudaEvent_t* events) {
    const int flags = ctx->l2_prefetch != 0 ? qb::QB_SWEEP_L2_PREFETCH : 0;
    const int streams = events ? 1 : std::min<int>(ctx->sweep_streams, b.batch / 4);
    const bool pdl = !events && (b.pdl || ctx->pdl >= 2);  // (event-timed runs measure every sweep on its own)
    if (streams > 1) {
        // circuits per group: by default the batch is cut into one group per stream; QB_SWEEP_GROUP = c makes groups of c circuits
        // that the streams take turns on (stream i runs groups i, i + streams, ... one after the other, each group all its sweeps
        // back to back) -- with small groups the states in flight stay L2-resident between their sweeps
        const int per = ctx->sweep_group > 0 ? std::min(ctx->sweep_group, b.batch) : (b.batch + streams - 1) / streams;
        const int groups = (b.batch + per - 1) / per;
        QB_CUDA(cudaEventRecord(ctx->fork_event, ctx->stream));  // bind_kernel (and uploads) done before any group starts
        const int fuse = b.fuse_expect ? (b.skip_final_store ? 2 : 1) : 0;
        for (int i = 0; i < streams; ++i) QB_CUDA(cudaStreamWaitEvent(ctx->aux_streams[i], ctx->fork_event, 0));
        for (int g = 0; g < groups; ++g) {
            const int lo = g * per, hi = std::min(b.batch, lo + per);
            cudaStream_t st = ctx->aux_streams[g % streams];
            for (int s = 0; s < b.max_sweeps; ++s) {
                const int active = std::min(b.active[s], hi) - lo;  // entries are sorted by descending sweep count
                if (active <= 0) break;
                dim3 grid(unsigned(b.n_tiles >> b.tiles_log2), unsigned(active));
                launch_kernel(qb::sweep_kernel<T, R, K, Idx>, grid, dim3(1 << (K - R)), qb::sweep_smem_bytes<T, R, K>(), st, pdl && s > 0,
                              b.entries.as<qb::BatchEntry>() + lo, s, b.n_eff, fuse, b.tiles_log2, flags);
                QB_TRY(check_launch(ctx, "sweep_kernel"));
            }
        }
        for (int i = 0; i < streams; ++i) {
            QB_CUDA(cudaEventRecord(ctx->join_events[i], ctx->aux_streams[i]));
            QB_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->join_events[i], 0));
        }
        return QB_OK;
    }
    for (int s = 0; s < b.max_sweeps; ++s) {
        // every CTA stages its circuit's sweep program once and walks 2^tiles_log2 consecutive tiles with it
        dim3 grid(unsigned(b.n_tiles >> b.tiles_log2), unsigned(b.active[s]));
        if (events) QB_CUDA(cudaEventRecord(events[2 * s], ctx->stream));
        // (the first sweep follows bind_kernel in this stream)
        launch_kernel(qb::sweep_kernel<T, R, K, Idx>, grid, dim3(1 << (K - R)), qb::sweep_smem_bytes<T, R, K>(), ctx->stream, pdl,
                      b.entries.as<qb::BatchEntry>(), s, b.n_eff, b.fuse_expect ? (b.skip_final_store ? 2 : 1) : 0, b.tiles_log2, flags);
        QB_TRY(check_launch(ctx, "sweep_kernel"));
        if (events) QB_CUDA(cudaEventRecord(events[2 * s + 1], ctx->stream));
    }
    return QB_OK;
}

int launch_circuits(qb_context* ctx, DeviceBatch& b, cudaEvent_t* events) {
    qb::bind_kernel<<<b.batch, 128, 0, ctx->stream>>>(b.entries.as<qb::BatchEntry>());
    QB_TRY(check_launch(ctx, "bind_kernel"));
    // amplitude indices fit 32 bits up to 31 local qubits: cheaper address arithmetic for the common sizes
#define QB_DISPATCH(R_, K_)                                                                                        \
    if (b.reg_bits == R_ && b.tile_bits == K_) {                                                                   \
        if (b.n_eff <= 31 && !ctx->force_idx64)                                                                    \
            return b.dtype == QB_C128 ? launch_sweeps_t<double, R_, K_, uint32_t>(ctx, b, events)                  \
                                      : launch_sweeps_t<float, R_, K_, uint32_t>(ctx, b, events);                  \
        return b.dtype == QB_C128 ? launch_sweeps_t<double, R_, K_, uint64_t>(ctx, b, events)                      \
                                  : launch_sweeps_t<float, R_, K_, uint64_t>(ctx, b, events);                      \
    }
    QB_DISPATCH(4, 11)
    QB_DISPATCH(4, 12)
    QB_DISPATCH(3, 11)
#undef QB_DISPATCH
    return fail(QB_ERR_INVALID, "unsupported tile / register bit combination");
}

// expectation of one resident state with the generic (non-fused) kernels; result accumulated into d_out[0]
template <typename T>
int expectation_state_t(qb_context* ctx, const Ham& ham, const void* d_state, int n_eff, uint64_t index_offset, double* d_partials,
                        double* d_out) {
    using C = typename qb::Cx<T>::type;
    const uint64_t size = uint64_t(1) << n_eff;
    const int blocks = int(std::min<uint64_t>(1024, std::max<uint64_t>(1, size / 256)));
    bool first = true;
    if (ham.table.p && ham.table_n_eff == n_eff && index_offset == 0) {
        qb::expect_table_kernel<T><<<blocks, 256, 0, ctx->stream>>>(static_cast<const C*>(d_state), size, ham.table.as<double>(), size, d_partials, 0);
        QB_TRY(check_launch(ctx, "expect_table_kernel"));
        qb::reduce_partials_kernel<<<1, 256, 0, ctx->stream>>>(d_partials, blocks, blocks, d_out, 0);
        QB_TRY(check_launch(ctx, "reduce_partials_kernel"));
        first = false;
    }
    // non-diagonal groups scheduled into tile sweeps: one read of the state per sweep of groups (usable on a shard as long as
    // every tile qubit is local; z masks may reach rank bits, they enter through index_offset)
    std::vector<char> done(ham.groups.size(), 0);
    if (!ham.tile_sweeps.empty() && n_eff >= qb::kExpTileBits) {
        const size_t tiles = size_t(1) << (n_eff - qb::kExpTileBits);
        const size_t smem = sizeof(C) << qb::kExpTileBits;
        for (size_t si = 0; si < ham.tile_sweeps.size(); ++si) {
            const auto& sw = ham.tile_sweeps[si];
            bool local = true;
            for (int i = 0; i < qb::kExpTileBits; ++i) local = local && sw.tile_qubits[i] < n_eff;
            if (!local) continue;
            qb::expect_tile_kernel<T><<<dim3(unsigned(tiles), 1), 256, smem, ctx->stream>>>(
                static_cast<const C*>(d_state), size, n_eff, index_offset, sw, ham.tile_groups.as<qb::ExpTileGroup>(), ham.tile_z.as<uint64_t>(),
                ham.tile_wr.as<double>(), ham.tile_wi.as<double>(), d_partials, tiles);
            QB_TRY(check_launch(ctx, "expect_tile_kernel"));
            qb::reduce_partials_kernel<<<1, 256, 0, ctx->stream>>>(d_partials, int64_t(tiles), int64_t(tiles), d_out, first ? 0 : 1);
            QB_TRY(check_launch(ctx, "reduce_partials_kernel"));
            first = false;
            for (int gi : ham.tile_sweep_groups[si]) done[gi] = 1;
        }
    }
    for (size_t gi = 0; gi < ham.groups.size(); ++gi) {
        const auto& g = ham.groups[gi];
        if (done[gi]) continue;
        if (g->xmask == 0 && !first && ham.table.p && ham.table_n_eff == n_eff && index_offset == 0) continue;  // diagonal part already taken from the table
        if (g->xmask >> n_eff) return fail(QB_ERR_INVALID, "Pauli term flips a qubit outside the local statevector");
        const bool stage = g->n_terms <= kMaxStagedTerms;
        const size_t smem = stage ? size_t(g->n_terms) * (sizeof(uint64_t) + 2 * sizeof(double)) : 0;
        qb::expect_group_kernel<T><<<blocks, 256, smem, ctx->stream>>>(static_cast<const C*>(d_state), size, size, index_offset, g->xmask,
                                                                       g->z.as<uint64_t>(), g->wr.as<double>(), g->wi.as<double>(),
                                                                       g->n_terms, stage ? 1 : 0, d_partials, 0);
        QB_TRY(check_launch(ctx, "expect_group_kernel"));
        qb::reduce_partials_kernel<<<1, 256, 0, ctx->stream>>>(d_partials, blocks, blocks, d_out, first ? 0 : 1);
        QB_TRY(check_launch(ctx, "reduce_partials_kernel"));
        first = false;
    }
    if (first) QB_CUDA(cudaMemsetAsync(d_out, 0, sizeof(double), ctx->stream));
    return QB_OK;
}

// batched <H>: diagonal part from the fused sweep epilogue / table / on-the-fly group, non-diagonal groups tile-fused
template <typename T> int launch_expectation_t(qb_context* ctx, DeviceBatch& b) {
    using C = typename qb::Cx<T>::type;
    const Ham& ham = *b.ham;
    const uint64_t size = uint64_t(1) << b.n_eff;
    const C* states = b.states.as<C>();
    double* partials = b.partials.as<double>();
    double* out = b.out_mapped ? b.out_mapped : b.out.as<double>();
    bool have = false;  // does `out` already hold a value to accumulate onto?
    auto reduce = [&](int64_t count, bool pdl = false) -> int {
        launch_kernel(qb::reduce_partials_kernel, dim3(unsigned(b.batch)), dim3(256), 0, ctx->stream, pdl, static_cast<const double*>(partials),
                      int64_t(b.partial_stride), count, out, have ? 1 : 0);
        have = true;
        return check_launch(ctx, "reduce_partials_kernel");
    };
    const int blocks = int(std::min<uint64_t>(1024, std::max<uint64_t>(1, size / 256)));
    // ---- diagonal part
    if (b.fuse_expect) {
        QB_TRY(reduce(int64_t(b.n_tiles >> b.tiles_log2), b.pdl));  // right behind the last sweep of the chain
    } else if (ham.n_diag > 0) {
        const bool table = ham.table.p && ham.table_n_eff == b.n_eff;
        const Group* dg = ham.groups.front().get();  // the x == 0 group is stored first
        const dim3 grid(unsigned(blocks), unsigned(b.batch));  // one launch for the whole batch
        if (table) {
            qb::expect_table_kernel<T><<<grid, 256, 0, ctx->stream>>>(states, size, ham.table.as<double>(), size, partials, b.partial_stride);
        } else {
            const bool stage = dg->n_terms <= kMaxStagedTerms;
            qb::expect_group_kernel<T><<<grid, 256, stage ? size_t(dg->n_terms) * (sizeof(uint64_t) + 2 * sizeof(double)) : 0, ctx->stream>>>(
                states, size, size, 0, 0, dg->z.as<uint64_t>(), dg->wr.as<double>(), dg->wi.as<double>(), dg->n_terms, stage ? 1 : 0, partials,
                b.partial_stride);
        }
        QB_TRY(check_launch(ctx, "diagonal expectation kernel"));
        QB_TRY(reduce(blocks));
    }
    // ---- non-diagonal groups that fit a tile: one read of every state per tile sweep
    const bool tiled = !ham.tile_sweeps.empty() && ham.tile_n_eff == b.n_eff;  // (padding differs only below 12 qubits)
    if (tiled) {
        const size_t tiles = size_t(1) << (b.n_eff - qb::kExpTileBits);
        const size_t smem = sizeof(C) << qb::kExpTileBits;
        for (const auto& sw : ham.tile_sweeps) {
            dim3 grid(unsigned(tiles), unsigned(b.batch));
            qb::expect_tile_kernel<T><<<grid, 256, smem, ctx->stream>>>(states, size, b.n_eff, 0, sw, ham.tile_groups.as<qb::ExpTileGroup>(),
                                                                        ham.tile_z.as<uint64_t>(), ham.tile_wr.as<double>(),
                                                                        ham.tile_wi.as<double>(), partials, b.partial_stride);
            QB_TRY(check_launch(ctx, "expect_tile_kernel"));
            QB_TRY(reduce(int64_t(tiles)));
        }
    }
    // ---- x masks wider than a tile: generic two-read kernel per group
    std::vector<int> generic = ham.generic_groups;
    if (!tiled)
        for (size_t gi = 0; gi < ham.groups.size(); ++gi)
            if (ham.groups[gi]->xmask != 0 && std::find(generic.begin(), generic.end(), int(gi)) == generic.end()) generic.push_back(int(gi));
    for (int gi : generic) {
        const Group* g = ham.groups[gi].get();
        if (g->xmask >> b.n_eff) return fail(QB_ERR_INVALID, "Pauli term flips a qubit outside the statevector");
        const bool stage = g->n_terms <= kMaxStagedTerms;
        qb::expect_group_kernel<T><<<dim3(unsigned(blocks), unsigned(b.batch)), 256, stage ? size_t(g->n_terms) * (sizeof(uint64_t) + 2 * sizeof(double)) : 0,
                                     ctx->stream>>>(states, size, size, 0, g->xmask, g->z.as<uint64_t>(), g->wr.as<double>(), g->wi.as<double>(), g->n_terms,
                                                    stage ? 1 : 0, partials, b.partial_stride);
        QB_TRY(check_launch(ctx, "expect_group_kernel"));
        QB_TRY(reduce(blocks));
    }
    if (!have) QB_TRY(reduce(0));  // no terms at all: zeros (a kernel, `out` may be mapped host memory)
    return QB_OK;
}

int launch_expectation(qb_context* ctx, DeviceBatch& b) {
    if (!b.ham) return fail(QB_ERR_INVALID, "batch was created without a Hamiltonian");
    return with_dtype(b.dtype, [&](auto t) { return launch_expectation_t<decltype(t)>(ctx, b); });
}

int batch_read(qb_context* ctx, DeviceBatch& b, double* out_values) {
    QB_TRY(ctx->pin_out.reserve(sizeof(double) * size_t(b.batch)));
    QB_CUDA(cudaMemcpyAsync(ctx->pin_out.p, b.out.p, sizeof(double) * size_t(b.batch), cudaMemcpyDeviceToHost, ctx->stream));
    QB_CUDA(cudaStreamSynchronize(ctx->stream));
    scatter_rows(out_values, ctx->pin_out.p, b.order, sizeof(double));
    return QB_OK;
}

void drop_single_graphs(qb_context* ctx, int64_t plan_id, int64_t ham_id) {
    for (auto it = ctx->single_graphs.begin(); it != ctx->single_graphs.end();) {
        bool hit = (plan_id && std::get<0>(it->first) == plan_id) || (ham_id && std::get<1>(it->first) == ham_id);
        if (!hit && plan_id) {  // a prefixed plan whose prefix goes away is rebuilt on next use as well
            Plan* pl = find_plan(ctx, std::get<0>(it->first));
            hit = pl && pl->prefix_id == plan_id;
        }
        if (hit) {
            ctx->single_graph_bytes -= it->second->state_bytes;
            it = ctx->single_graphs.erase(it);
        } else {
            ++it;
        }
    }
}

// qb_evaluate_expectation of ONE circuit at 1 .. kMaxGraphCopies parameter points (the optimizer loop's calls: SPSA evaluates
// theta +- c delta together) through a cached CUDA graph.  Returns QB_OK with *handled = false when the graph path does not
// apply (disabled, states too large to keep resident per circuit).
constexpr int kMaxGraphCopies = 4;  // (from 8 entries on the sweep launches fork into stream groups)
int evaluate_single_graph(qb_context* ctx, int64_t plan_id, Plan* pl, Ham* ham, int64_t ham_id, int copies, const double* params,
                          const int64_t* param_offsets, double* out_values, bool* handled) {
    *handled = false;
    const size_t state_bytes = (size_t(1) << pl->n_eff) * amp_bytes(pl->dtype) * size_t(copies);
    const size_t budget = std::min<size_t>(size_t(4) << 30, workspace_limit_of(ctx) / 8);
    if (!ctx->use_graphs || state_bytes > budget / 4) return QB_OK;
    for (int i = 0; i < copies; ++i)
        if (param_offsets[i + 1] - param_offsets[i] != pl->n_params)
            return fail(QB_ERR_INVALID, "entry " + std::to_string(i) + ": got " + std::to_string(param_offsets[i + 1] - param_offsets[i]) +
                                            " parameter values, circuit has " + std::to_string(pl->n_params) + " parameters");
    const auto key = std::make_tuple(plan_id, ham_id, copies);
    auto it = ctx->single_graphs.find(key);
    if (it == ctx->single_graphs.end()) {
        while (!ctx->single_graphs.empty() && (ctx->single_graph_bytes + state_bytes > budget || ctx->single_graphs.size() >= 256)) {
            auto victim = ctx->single_graphs.begin();
            for (auto j = ctx->single_graphs.begin(); j != ctx->single_graphs.end(); ++j)
                if (j->second->last_use < victim->second->last_use) victim = j;
            QB_CUDA(cudaStreamSynchronize(ctx->stream));
            ctx->single_graph_bytes -= victim->second->state_bytes;
            ctx->single_graphs.erase(victim);
        }
        auto sg = std::make_unique<SingleGraph>();
        sg->state_bytes = state_bytes;
        sg->pin_params.mapped = sg->pin_out.mapped = ctx->zero_copy;
        const size_t params_bytes = sizeof(double) * size_t(pl->n_params) * size_t(copies), out_bytes = sizeof(double) * size_t(copies);
        QB_TRY(sg->pin_params.reserve(std::max<size_t>(params_bytes, 16)));
        QB_TRY(sg->pin_out.reserve(out_bytes));
        if (ctx->zero_copy) {
            // no copy nodes: bind_kernel reads the (few) parameters from mapped pinned memory, the reduction writes the value there
            sg->batch.params_mapped = static_cast<const double*>(sg->pin_params.device_ptr());
            sg->batch.out_mapped = static_cast<double*>(sg->pin_out.device_ptr());
        }
        const std::vector<int64_t> ids(size_t(copies), plan_id);
        QB_TRY(build_batch(ctx, sg->batch, copies, ids.data(), ham, nullptr, 1, 0));  // (also computes a cached prefix state, uncaptured)
        QB_CUDA(cudaStreamSynchronize(ctx->stream));
        // capture: [parameter upload] -> bind -> sweeps -> reduction(s) -> [result download]; with programmatic dependent launches
        // first, in the ordinary way if the driver refuses those inside a capture
        for (int attempt = (ctx->pdl >= 1 ? 0 : 1); attempt < 2 && !sg->exec; ++attempt) {
            sg->batch.pdl = attempt == 0;
            cudaGraph_t graph = nullptr;
            QB_CUDA(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
            int rc = QB_OK;
            if (pl->n_params && !sg->batch.params_mapped &&
                cudaMemcpyAsync(sg->batch.params.p, sg->pin_params.p, params_bytes, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess)
                rc = fail(QB_ERR_CUDA, "graph capture: parameter upload");
            if (rc == QB_OK) rc = launch_circuits(ctx, sg->batch, nullptr);
            if (rc == QB_OK) rc = launch_expectation(ctx, sg->batch);
            if (rc == QB_OK && !sg->batch.out_mapped &&
                cudaMemcpyAsync(sg->pin_out.p, sg->batch.out.p, out_bytes, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess)
                rc = fail(QB_ERR_CUDA, "graph capture: result download");
            cudaError_t ce = cudaStreamEndCapture(ctx->stream, &graph);
            if (rc == QB_OK && ce == cudaSuccess && graph) ce = cudaGraphInstantiate(&sg->exec, graph, 0);
            if (graph) cudaGraphDestroy(graph);
            if (rc != QB_OK || ce != cudaSuccess) {
                cudaGetLastError();
                sg->exec = nullptr;
                if (attempt == 0) continue;
                ctx->use_graphs = false;  // capture is not available here: fall back to plain launches for good
                return rc != QB_OK ? rc : QB_OK;
            }
        }
        ctx->single_graph_bytes += state_bytes;
        it = ctx->single_graphs.emplace(key, std::move(sg)).first;
    }
    SingleGraph& sg = *it->second;
    sg.last_use = ++ctx->use_clock;
    for (int i = 0; i < copies && pl->n_params; ++i)  // entry i's parameters live at param_begin[i] (caller order)
        std::memcpy(static_cast<double*>(sg.pin_params.p) + sg.batch.param_begin[i], params + param_offsets[i], sizeof(double) * size_t(pl->n_params));
    QB_CUDA(cudaGraphLaunch(sg.exec, ctx->stream));
    ctx->launches += sg.batch.max_sweeps + 2;  // bind + sweeps + reduction(s), as counted for plain launches
    QB_CUDA(cudaStreamSynchronize(ctx->stream));
    const volatile double* sorted = static_cast<const volatile double*>(sg.pin_out.p);
    for (int pos = 0; pos < copies; ++pos) out_values[sg.batch.order[pos]] = sorted[pos];
    *handled = true;
    return QB_OK;
}

size_t max_batch_for(qb_context* ctx, const Plan* pl) {
    const size_t state_bytes = (size_t(1) << pl->n_eff) * amp_bytes(pl->dtype);
    return std::min<size_t>(65535, std::max<size_t>(1, workspace_limit_of(ctx) / state_bytes));  // 65535: grid.y of the batched launches
}

// E(k) of the Hamiltonian's diagonal terms for k < 2^n_eff into `table` (asynchronous on the context's stream)
int fill_diag_table(qb_context* ctx, const Ham& ham, double* table, int n_eff) {
    const uint64_t size = uint64_t(1) << n_eff;
    if (ham.n_diag == 0) {
        QB_CUDA(cudaMemsetAsync(table, 0, sizeof(double) * size, ctx->stream));
        return QB_OK;
    }
    const int blocks = int(std::min<uint64_t>(uint64_t(ctx->sm_count) * 8, std::max<uint64_t>(1, size / 256)));
    for (int lo = 0; lo < ham.n_diag; lo += kTableTermChunk) {  // term order is kept: chunk after chunk accumulates onto the table
        const int cnt = std::min(kTableTermChunk, ham.n_diag - lo);
        qb::diag_table_kernel<<<blocks, 256, size_t(cnt) * (sizeof(uint64_t) + sizeof(double)), ctx->stream>>>(
            table, size, 0, ham.diag_z.as<uint64_t>() + lo, ham.diag_c.as<double>() + lo, cnt, lo ? 1 : 0);
        QB_TRY(check_launch(ctx, "diag_table_kernel"));
    }
    return QB_OK;
}

// Build (once per Hamiltonian and state width) what qb_evaluate_cvar reads: E(k) in basis order (8 B per amplitude); with `sorted`
// also a stable ascending radix sort of (E(k), k) -> perm (sorted position -> k, 4 B) and E_sorted (8 B).  CUB's radix sort is
// stable and treats -0.0 == +0.0, which is numpy.argsort(kind="stable") on float64.  The sort needs the input indices and CUB's
// sort storage for a moment.
int ensure_cvar_order(qb_context* ctx, Ham& ham, int n_eff, bool sorted) {
    // perm holds basis indices as uint32: above 2^32 entries they would wrap, whatever the workspace holds
    if (sorted && n_eff > 32)
        return fail(QB_ERR_INVALID, "the sorted CVaR order of a " + std::to_string(n_eff) +
                                        "-qubit state needs basis indices wider than 32 bits; only alpha close to 1 (basis order) is supported above 32 qubits");
    const uint64_t size = uint64_t(1) << n_eff;
    const size_t limit = workspace_limit_of(ctx);
    if (ham.cvar_energy_n_eff != n_eff) {
        if (sizeof(double) * size > limit)
            return fail(QB_ERR_MEMORY, "the CVaR energies of a " + std::to_string(n_eff) + "-qubit Hamiltonian need " +
                                           std::to_string(sizeof(double) * size) + " bytes, the workspace is " + std::to_string(limit) + " bytes");
        ham.cvar_energy_n_eff = ham.cvar_order_n_eff = 0;
        QB_TRY(ham.cvar_energy.reserve(sizeof(double) * size));
        QB_TRY(fill_diag_table(ctx, ham, ham.cvar_energy.as<double>(), n_eff));
        QB_CUDA(cudaStreamSynchronize(ctx->stream));
        ham.cvar_energy_n_eff = n_eff;
    }
    if (!sorted || ham.cvar_order_n_eff == n_eff) return QB_OK;
    size_t sort_bytes = 0;
    QB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, static_cast<const double*>(nullptr), static_cast<double*>(nullptr),
                                            static_cast<const uint32_t*>(nullptr), static_cast<uint32_t*>(nullptr), int64_t(size), 0,
                                            int(sizeof(double) * 8), ctx->stream));
    const size_t index_at = (sort_bytes + 255) & ~size_t(255);
    const size_t kept = (sizeof(double) * 2 + sizeof(uint32_t)) * size, need = kept + index_at + sizeof(uint32_t) * size;
    if (need > limit)
        return fail(QB_ERR_MEMORY, "the CVaR order data of a " + std::to_string(n_eff) + "-qubit Hamiltonian needs " + std::to_string(need) +
                                       " bytes to build (" + std::to_string(kept) + " kept), the workspace is " + std::to_string(limit) + " bytes");
    QB_TRY(ham.cvar_sorted.reserve(sizeof(double) * size));
    QB_TRY(ham.cvar_perm.reserve(sizeof(uint32_t) * size));
    DevBuf temp;
    QB_TRY(temp.reserve(index_at + sizeof(uint32_t) * size));
    uint32_t* index = reinterpret_cast<uint32_t*>(static_cast<unsigned char*>(temp.p) + index_at);
    const int blocks = int(std::min<uint64_t>(uint64_t(ctx->sm_count) * 8, std::max<uint64_t>(1, size / 256)));
    qb::iota_u32_kernel<<<blocks, 256, 0, ctx->stream>>>(index, size);
    int rc = check_launch(ctx, "iota_u32_kernel");
    if (rc == QB_OK) {
        cudaError_t e = cub::DeviceRadixSort::SortPairs(temp.p, sort_bytes, ham.cvar_energy.as<double>(), ham.cvar_sorted.as<double>(), index,
                                                        ham.cvar_perm.as<uint32_t>(), int64_t(size), 0, int(sizeof(double) * 8), ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = fail(QB_ERR_CUDA, std::string("cub::DeviceRadixSort::SortPairs: ") + cudaGetErrorString(e));
    }
    temp.release();
    if (rc == QB_OK) ham.cvar_order_n_eff = n_eff;
    return rc;
}

// Pauli strings grouped by x mask, groups in first-appearance order: xs[g] and the string indices of each group
int group_by_xmask(int n_qubits, int n_terms, const uint64_t* x_masks, const uint64_t* z_masks, std::vector<uint64_t>& xs,
                   std::vector<std::vector<int>>& members) {
    for (int t = 0; t < n_terms; ++t) {
        if ((x_masks[t] | z_masks[t]) >> n_qubits) return fail(QB_ERR_INVALID, "Pauli term acts outside the register");
        size_t g = 0;
        for (; g < xs.size(); ++g)
            if (xs[g] == x_masks[t]) break;
        if (g == xs.size()) xs.push_back(x_masks[t]), members.emplace_back();
        members[g].push_back(t);
    }
    return QB_OK;
}

// Schedule x-mask groups into tile sweeps: every sweep takes, in order, the pending groups whose flipped qubits still fit one
// 2^kExpTileBits tile next to qubits 0 .. QB_LOW_BITS-1; a group that does not fit a tile on its own is left to a generic kernel.
// Group records of the sweeps are laid out sweep after sweep, in `sweep_groups` order (group_begin / group_end count them).
struct TilePlan {
    std::vector<qb::ExpTileSweep> sweeps;
    std::vector<std::vector<int>> sweep_groups;  // group indices of every sweep
    std::vector<uint32_t> xloc;                  // per group: x mask in the tile-local bit positions of its sweep
    std::vector<int> generic;                    // groups whose x mask does not fit a tile
};

TilePlan plan_tile_sweeps(int n_eff, const std::vector<uint64_t>& xmask, std::vector<int> pending) {
    const int K = qb::kExpTileBits, low = QB_LOW_BITS;
    TilePlan tp;
    tp.xloc.assign(xmask.size(), 0);
    int n_records = 0;
    while (!pending.empty()) {
        uint64_t tile = (uint64_t(1) << low) - 1;
        std::vector<int> chosen, rest;
        for (int g : pending) {
            const uint64_t want = tile | xmask[g];
            if (__builtin_popcountll(want) <= K) tile = want, chosen.push_back(g);
            else rest.push_back(g);
        }
        if (chosen.empty()) {  // the first pending group alone does not fit a tile: generic kernel
            tp.generic.push_back(pending.front());
            pending.erase(pending.begin());
            continue;
        }
        for (int q = 0; __builtin_popcountll(tile) < K; ++q) tile |= uint64_t(1) << q;
        qb::ExpTileSweep sw{};
        int pos_of[64];
        for (int q = 0, i = 0; q < n_eff; ++q)
            if ((tile >> q) & 1) pos_of[q] = i, sw.tile_qubits[i++] = q;
        sw.group_begin = n_records;
        for (int g : chosen)
            for (int q = 0; q < n_eff; ++q)
                if ((xmask[g] >> q) & 1) tp.xloc[g] |= 1u << pos_of[q];
        n_records += int(chosen.size());
        sw.group_end = n_records;
        tp.sweeps.push_back(sw);
        tp.sweep_groups.push_back(chosen);
        pending = rest;
    }
    return tp;
}

Obs* find_obs(qb_context* ctx, int64_t id) {
    auto it = ctx->observables.find(id);
    return it == ctx->observables.end() ? nullptr : it->second.get();
}

// partial-sum scratch of one term-resolved launch: terms beyond it are evaluated in further launches over the same state
constexpr size_t kTermPartialBytes = size_t(256) << 20;

// <P_t> of every string of `ob` for the n resident states of `b` into d_terms[pos * n_terms + slot]
template <typename T>
int launch_terms_t(qb_context* ctx, const DeviceBatch& b, const Obs& ob, double* d_partials, size_t partial_bytes, double* d_terms) {
    using C = typename qb::Cx<T>::type;
    const int n = b.batch;
    const uint64_t size = uint64_t(1) << b.n_eff;
    const C* states = b.states.as<C>();
    // terms [lo, hi) in pieces whose partials (n states x terms x count) fit the scratch; a term's value does not depend on the piece
    auto pieces = [&](int lo, int hi, uint64_t count, const std::function<int(int, int)>& run) -> int {
        const int per = int(std::max<uint64_t>(1, std::min<uint64_t>(uint64_t(hi - lo), partial_bytes / (sizeof(double) * count * uint64_t(n)))));
        for (int t0 = lo; t0 < hi; t0 += per) {
            const int t1 = std::min(hi, t0 + per);
            QB_TRY(run(t0, t1));
            qb::reduce_term_partials_kernel<<<dim3(unsigned(t1 - t0), unsigned(n)), 256, 0, ctx->stream>>>(
                d_partials, int64_t(count), t1 - t0, ob.sign.as<double>(), t0, d_terms, ob.n_terms);
            QB_TRY(check_launch(ctx, "reduce_term_partials_kernel"));
        }
        return QB_OK;
    };
    const uint64_t tiles = size >> qb::kExpTileBits;
    const size_t smem = sizeof(C) << qb::kExpTileBits;
    for (size_t s = 0; s < ob.tile_sweeps.size(); ++s) {
        const auto& sw = ob.tile_sweeps[s];
        QB_TRY(pieces(ob.sweep_terms[s].first, ob.sweep_terms[s].second, tiles, [&](int t0, int t1) {
            qb::expect_terms_tile_kernel<T><<<dim3(unsigned(tiles), unsigned(n)), 256, smem, ctx->stream>>>(
                states, size, b.n_eff, sw, ob.groups.as<qb::TermGroup>(), ob.z.as<uint64_t>(), ob.im.as<int8_t>(), t0, t1, d_partials);
            return check_launch(ctx, "expect_terms_tile_kernel");
        }));
    }
    const uint64_t blocks = std::min<uint64_t>(1024, std::max<uint64_t>(1, size / 256));
    for (const auto& g : ob.generic) {
        if (g.xmask >> b.n_eff) return fail(QB_ERR_INVALID, "Pauli term flips a qubit outside the statevector");
        QB_TRY(pieces(g.term_begin, g.term_end, blocks, [&](int t0, int t1) {
            qb::expect_terms_group_kernel<T><<<dim3(unsigned(blocks), unsigned(n)), 256, 0, ctx->stream>>>(
                states, size, size, g.xmask, ob.z.as<uint64_t>(), ob.im.as<int8_t>(), t0, t1, t0, t1 - t0, d_partials);
            return check_launch(ctx, "expect_terms_group_kernel");
        }));
    }
    return QB_OK;
}

// shots from each of the n states (stride `size`): chunk probabilities, their prefix sums, one search per uniform; indices stay
// below `valid_size`
template <typename T>
int launch_sampling_t(qb_context* ctx, const typename qb::Cx<T>::type* states, uint64_t size, int n, uint64_t valid_size, const double* d_uniforms,
                      int shots, double* d_chunks, int64_t* d_indices) {
    const uint64_t n_chunks = size >> qb::kChunkBits;
    dim3 cgrid(unsigned(std::min<uint64_t>((n_chunks + 7) / 8, 2048)), unsigned(n));
    dim3 sgrid(unsigned((shots + 7) / 8), unsigned(n));
    qb::chunk_prob_kernel<T><<<cgrid, 256, 0, ctx->stream>>>(states, size, n_chunks, d_chunks);
    QB_TRY(check_launch(ctx, "chunk_prob_kernel"));
    qb::scan_chunks_kernel<<<n, 1024, 0, ctx->stream>>>(d_chunks, n_chunks);
    QB_TRY(check_launch(ctx, "scan_chunks_kernel"));
    qb::sample_kernel<T><<<sgrid, 256, 0, ctx->stream>>>(states, size, d_chunks, n_chunks, valid_size, d_uniforms, shots, d_indices);
    return check_launch(ctx, "sample_kernel");
}

// Every plan of a call whose chunks share one operator's device data must act on the operator's `n_qubits` and share the first
// plan's state width and dtype.  `acts`: the operator's subject and verb in the message; `call`: the call's name.
int check_plans(qb_context* ctx, int batch, const int64_t* plan_ids, int n_qubits, const char* acts, const char* call, const Plan** first) {
    for (int i = 0; i < batch; ++i) {
        const Plan* pl = find_plan(ctx, plan_ids[i]);
        if (!pl) return fail(QB_ERR_NOT_FOUND, "unknown plan id " + std::to_string(plan_ids[i]));
        if (i == 0) *first = pl;
        if (pl->n_qubits != n_qubits)
            return fail(QB_ERR_INVALID, std::string(acts) + " on " + std::to_string(n_qubits) + " qubits, circuit " + std::to_string(i) + " on " +
                                            std::to_string(pl->n_qubits));
        if (pl->n_eff != (*first)->n_eff || pl->dtype != (*first)->dtype)
            return fail(QB_ERR_INVALID, std::string("all plans of one ") + call + " call must share state width and dtype");
    }
    return QB_OK;
}

// Runs `batch` circuits through the context's one-shot batch, `chunk` at a time; after each chunk's launches
// readout(b, lo) reads its resident states, which hold caller entries lo + b.order[pos] in sorted device order.
template <typename ReadOut>
int run_oneshot(qb_context* ctx, int batch, const int64_t* plan_ids, const double* params, const int64_t* param_offsets, const Ham* ham, int chunk,
                ReadOut&& readout) {
    for (int lo = 0; lo < batch; lo += chunk) {
        DeviceBatch& b = ctx->oneshot;
        QB_TRY(build_batch(ctx, b, std::min(chunk, batch - lo), plan_ids + lo, ham, nullptr, 1, 0));
        QB_TRY(batch_upload_params(ctx, b, params, param_offsets + lo));
        QB_TRY(launch_circuits(ctx, b, nullptr));
        QB_TRY(readout(b, lo));
    }
    return QB_OK;
}

// f(uint32_t()) where the sweep kernels use 32-bit amplitude indices (up to 31 qubits, unless forced wide), f(uint64_t()) above
template <typename F> int with_index_width(const qb_context* ctx, int n_bits, F&& f) {
    return n_bits <= 31 && !ctx->force_idx64 ? f(uint32_t()) : f(uint64_t());
}

// ---- top states: validation, pass arguments, grids ----
constexpr int64_t kTopMaxStates = int64_t(1) << 20;
static_assert(sizeof(qb_top_select) == 88, "qb_top_select is mirrored by _native.TopSelect");

int check_top_limits(int64_t max_states, double min_probability) {
    if (max_states < 1 || max_states > kTopMaxStates) return fail(QB_ERR_INVALID, "max_states must be in 1..2^20, got " + std::to_string(max_states));
    if (!std::isfinite(min_probability) || min_probability < 0.0) return fail(QB_ERR_INVALID, "min_probability must be finite and >= 0");
    return QB_OK;
}

// a select state as qb_top_select_init / _pick leave it, and a bit map of distinct positions below 64 (null: the identity)
int check_top_state(const qb_top_select* s, const int32_t* positions, bool want_done) {
    if (!s) return fail(QB_ERR_INVALID, "null select state");
    if (s->n_qubits < 1 || s->n_qubits > 63 || s->p_free < 0 || s->p_free > 64 || s->p_free % qb::kSelBits || s->idx_hi < 0 ||
        s->idx_hi > s->n_qubits || (s->p_free && s->idx_hi != s->n_qubits))
        return fail(QB_ERR_INVALID, "malformed select state");
    if (bool(s->done) != want_done) return fail(QB_ERR_INVALID, want_done ? "the select is not done yet" : "the select is already done");
    if (positions) {
        uint64_t seen = 0;
        for (int q = 0; q < s->n_qubits; ++q) {
            const int p = positions[q];
            if (p < 0 || p > 63 || ((seen >> p) & 1)) return fail(QB_ERR_INVALID, "bad bit map: positions must be distinct and below 64");
            seen |= uint64_t(1) << p;
        }
    }
    return QB_OK;
}

int top_position(const int32_t* positions, int q) { return positions ? positions[q] : q; }

qb::TopSelectArgs top_select_args(const qb_top_select& s, const int32_t* positions, double min_probability, int entry) {
    qb::TopSelectArgs t{};
    qb::SelectArgs& a = t.sel;
    a.e_prefix = s.p_prefix, a.e_free = s.p_free;
    if (s.p_free > 0) {
        a.digit_kind = 0, a.bits = qb::kSelBits;
    } else {  // the probability key is fixed: logical index bits [lo, idx_hi), read at their physical positions
        const int lo = std::max(0, s.idx_hi - qb::kSelBits);
        a.digit_kind = 1, a.bits = s.idx_hi - lo;
        for (int j = 0; j < a.bits; ++j) a.pos[j] = top_position(positions, lo + j);
        for (int q = s.idx_hi; q < s.n_qubits; ++q) {
            a.idx_mask |= uint64_t(1) << top_position(positions, q);
            a.idx_value |= ((s.idx_prefix >> q) & 1) << top_position(positions, q);
        }
    }
    t.min_probability = min_probability, t.entry = entry;
    return t;
}

qb::TopCollectArgs top_collect_args(const qb_top_select& s, const int32_t* positions, double min_probability, int entry) {
    qb::TopCollectArgs a{};
    a.stop_key = s.stop_key, a.stop_index = s.stop_index, a.min_probability = min_probability, a.entry = entry;
    if (positions) {
        a.n_pos = s.n_qubits;
        for (int q = 0; q < s.n_qubits; ++q) a.pos[q] = int8_t(positions[q]);
    }
    return a;
}

// select grid: one wave of resident CTAs, fewer for small states (fixed by the device and the state size)
unsigned top_select_ctas(const qb_context* ctx, uint64_t size) {
    return unsigned(std::min<uint64_t>(uint64_t(ctx->sm_count) * 8, std::max<uint64_t>(1, size / (32 * qb::kSelWarps * qb::kTopUnroll * 4))));
}

// collect grid: contiguous segments of whole kTopTile steps, about four waves
unsigned top_collect_ctas(const qb_context* ctx, uint64_t size, uint64_t* seg) {
    const uint64_t want = std::min<uint64_t>(uint64_t(ctx->sm_count) * 32, std::max<uint64_t>(1, size / qb::kTopTile));
    *seg = ((size + want - 1) / want + qb::kTopTile - 1) / qb::kTopTile * qb::kTopTile;
    return unsigned((size + *seg - 1) / *seg);
}

// one select pass over `m` states (rows `stride` amplitudes apart): d_counts[r][b] for args[r]; copied to host_counts
template <typename T>
int top_select_pass_t(qb_context* ctx, const void* states, uint64_t stride, uint64_t size, int n_bits, uint64_t index_offset,
                      const qb::TopSelectArgs* host_args, int m, qb::TopSelectArgs* d_args, unsigned long long* d_counts, uint64_t* host_counts) {
    using C = typename qb::Cx<T>::type;
    const size_t count_bytes = sizeof(uint64_t) * qb::kSelBuckets * size_t(m);
    QB_CUDA(cudaMemcpyAsync(d_args, host_args, sizeof(qb::TopSelectArgs) * size_t(m), cudaMemcpyHostToDevice, ctx->stream));
    QB_CUDA(cudaMemsetAsync(d_counts, 0, count_bytes, ctx->stream));
    const dim3 grid(top_select_ctas(ctx, size), unsigned(m));
    QB_TRY(with_index_width(ctx, n_bits, [&](auto i) {
        using Idx = decltype(i);
        qb::top_select_kernel<T, Idx><<<grid, 32 * qb::kSelWarps, 0, ctx->stream>>>(static_cast<const C*>(states), stride, Idx(size), index_offset, d_args,
                                                                                     d_counts);
        return check_launch(ctx, "top_select_kernel");
    }));
    QB_TRY(ctx->pin_out.reserve(count_bytes));
    QB_CUDA(cudaMemcpyAsync(ctx->pin_out.p, d_counts, count_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    QB_CUDA(cudaStreamSynchronize(ctx->stream));
    std::memcpy(host_counts, ctx->pin_out.p, count_bytes);
    return QB_OK;
}

// the collect of `n` states: count pass, check of the totals against `expect`, store pass into rows of `capacity`
template <typename T>
int top_collect_t(qb_context* ctx, const void* states, uint64_t stride, uint64_t size, int n_bits, uint64_t index_offset,
                  const qb::TopCollectArgs* host_args, int n, qb::TopCollectArgs* d_args, uint32_t* d_cta, uint64_t capacity, int64_t* d_index,
                  double* d_prob, std::vector<uint64_t>& totals) {
    using C = typename qb::Cx<T>::type;
    uint64_t seg = 0;
    const unsigned n_cta = top_collect_ctas(ctx, size, &seg);
    QB_CUDA(cudaMemcpyAsync(d_args, host_args, sizeof(qb::TopCollectArgs) * size_t(n), cudaMemcpyHostToDevice, ctx->stream));
    const dim3 grid(n_cta, unsigned(n));
    for (int store = 0; store < 2; ++store) {
        QB_TRY(with_index_width(ctx, n_bits, [&](auto i) {
            using Idx = decltype(i);
            qb::top_collect_kernel<T, Idx><<<grid, qb::kTopCollectThreads, 0, ctx->stream>>>(static_cast<const C*>(states), stride, Idx(size), Idx(seg),
                                                                                           index_offset, d_args, d_cta, store, capacity, d_index, d_prob);
            return check_launch(ctx, "top_collect_kernel");
        }));
        if (store) break;
        const size_t cta_bytes = sizeof(uint32_t) * n_cta * size_t(n);
        QB_TRY(ctx->pin_out.reserve(cta_bytes));
        QB_CUDA(cudaMemcpyAsync(ctx->pin_out.p, d_cta, cta_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        QB_CUDA(cudaStreamSynchronize(ctx->stream));
        const uint32_t* c = static_cast<const uint32_t*>(ctx->pin_out.p);
        totals.assign(size_t(n), 0);
        for (int r = 0; r < n; ++r)
            for (unsigned i = 0; i < n_cta; ++i) totals[r] += c[size_t(r) * n_cta + i];
        for (int r = 0; r < n; ++r)
            if (totals[r] > capacity)
                return fail(QB_ERR_INVALID, "the collect found " + std::to_string(totals[r]) + " entries, more than the capacity of " + std::to_string(capacity));
    }
    return QB_OK;
}

int check_top_shard(qb_context* ctx, int dtype, int n_local, const void* d_state, double min_probability, const qb_top_select* sel,
                    const int32_t* positions, bool want_done) {
    if (!ctx || !d_state) return fail(QB_ERR_INVALID, "null argument");
    if (n_local < 8 || n_local > 36) return fail(QB_ERR_INVALID, "n_local out of range");
    if (dtype != QB_C128 && dtype != QB_C64) return fail(QB_ERR_INVALID, "dtype must be QB_C128 or QB_C64");
    QB_TRY(check_top_limits(1, min_probability));
    return check_top_state(sel, positions, want_done);
}

// ---- exact marginal probabilities ----
// The kernel arguments for measured bit positions pos[0..m) (distinct, below `limit`) of a state of 2^n_bits amplitudes whose
// indices are index_offset | k: positions >= n_bits are rank bits and read their value from index_offset.  The slice count
// (2^slice_bits items per measured-bit value) brings the items to about 2^kMargItemBits.
int marginal_args(int n_bits, uint64_t index_offset, int m, const int* pos, int limit, qb::MarginalArgs* out) {
    if (!pos) return fail(QB_ERR_INVALID, "null qubit list");
    if (m < 1 || m > qb::kMargMaxBits) return fail(QB_ERR_INVALID, "n_measured must be in 1.." + std::to_string(qb::kMargMaxBits) + ", got " + std::to_string(m));
    qb::MarginalArgs a{};
    int out_of[64];
    std::fill(out_of, out_of + 64, -1);
    for (int j = 0; j < m; ++j) {
        if (pos[j] < 0 || pos[j] >= limit || out_of[pos[j]] >= 0)
            return fail(QB_ERR_INVALID, "measured qubits must be distinct and in 0.." + std::to_string(limit - 1));
        out_of[pos[j]] = j;
    }
    for (int p = 0; p < 64; ++p) {
        const int j = out_of[p];
        if (p < 5) {
            if (j >= 0) a.lane_bin[p] = 1u << j;
            else if (p < n_bits) a.lane_sum |= 1u << p;
        } else if (p < n_bits) {
            if (j >= 0) a.h_pos[a.h_bits] = int8_t(p - 5), a.h_out[a.h_bits] = int8_t(j), ++a.h_bits;
            else a.v_pos[a.v_bits] = int8_t(p - 5), a.v_mask |= 1u << (p - 5), ++a.v_bits;
        } else if (j >= 0) {
            a.bin_fixed |= uint32_t((index_offset >> p) & 1) << j;
            a.fixed_mask |= 1u << j;
        }
    }
    a.m = m;
    a.slice_bits = std::min(a.v_bits, std::max(0, qb::kMargItemBits - a.h_bits));
    *out = a;
    return QB_OK;
}

// bytes of device scratch per state: the marginal, and the [bin][slice] partial rows when there are several slices
size_t marginal_scratch_bytes(const qb::MarginalArgs& a) {
    return (sizeof(double) << a.m) + (a.slice_bits ? sizeof(double) << (a.m + a.slice_bits) : 0);
}

// the marginals of `n` states (rows `stride` amplitudes apart) into d_out[n][2^m]; d_part: n rows of partials when sliced
template <typename T>
int marginal_t(qb_context* ctx, const void* states, uint64_t stride, int n, int n_bits, const qb::MarginalArgs& a, double* d_part, double* d_out) {
    using C = typename qb::Cx<T>::type;
    const uint64_t items = uint64_t(1) << (a.h_bits + a.slice_bits);
    const dim3 grid(unsigned(std::min<uint64_t>(uint64_t(ctx->sm_count) * 8, (items + qb::kMargWarps - 1) / qb::kMargWarps)), unsigned(n));
    double* dst = a.slice_bits ? d_part : d_out;
    // a shard's items only reach the bins of its own rank-bit pattern: the others are zero
    if (!a.slice_bits && a.fixed_mask) QB_CUDA(cudaMemsetAsync(d_out, 0, (sizeof(double) << a.m) * size_t(n), ctx->stream));
    QB_TRY(with_index_width(ctx, n_bits, [&](auto i) {
        using Idx = decltype(i);
        qb::marginal_kernel<T, Idx><<<grid, 32 * qb::kMargWarps, 0, ctx->stream>>>(static_cast<const C*>(states), stride, a, dst);
        return check_launch(ctx, "marginal_kernel");
    }));
    if (!a.slice_bits) return QB_OK;
    const int group_bits = std::min(8, std::max(5, a.slice_bits - 6));  // 32..256 threads per bin, 64 slices per thread below 256
    const int bins_per_block = 256 >> group_bits;
    const dim3 rgrid(unsigned(((uint64_t(1) << a.m) + bins_per_block - 1) / bins_per_block), unsigned(n));
    qb::marginal_reduce_kernel<<<rgrid, 256, 0, ctx->stream>>>(d_part, a.m, a.slice_bits, group_bits, a.fixed_mask, a.bin_fixed, d_out);
    return check_launch(ctx, "marginal_reduce_kernel");
}

}  // namespace

// =====================================================================================================
extern "C" {

const char* qb_last_error(void) { return g_last_error.c_str(); }

void qb_record_sizes(int32_t out[4]) {
    out[0] = int32_t(sizeof(qb_sweep));
    out[1] = int32_t(sizeof(qb_pass));
    out[2] = int32_t(sizeof(qb_pass_op));
    out[3] = int32_t(sizeof(qb_op_angles));
}

int qb_device_count(int* out) {
    if (!out) return fail(QB_ERR_INVALID, "out is null");
    int count = 0;
    QB_CUDA(cudaGetDeviceCount(&count));
    *out = count;
    return QB_OK;
}

int qb_context_create(int device, void* stream, qb_context** out) {
    if (!out) return fail(QB_ERR_INVALID, "out is null");
    int count = 0;
    QB_CUDA(cudaGetDeviceCount(&count));
    if (device < 0 || device >= count) return fail(QB_ERR_INVALID, "no CUDA device " + std::to_string(device));
    DeviceScope scope(device);
    if (scope.err != cudaSuccess) return fail(QB_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(scope.err));
    cudaDeviceProp prop;
    QB_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return fail(QB_ERR_CUDA, std::string("device '") + prop.name + "' is sm_" + std::to_string(prop.major) + std::to_string(prop.minor) +
                                     "; this library is built for sm_100a (B200) only");
    auto ctx = std::make_unique<qb_context>();
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    if (stream) {
        ctx->stream = static_cast<cudaStream_t>(stream);
    } else {
        QB_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        ctx->owns_stream = true;
    }
    {
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) ctx->default_workspace = free_b / 10 * 8;
    }
    QB_CUDA(cudaEventCreateWithFlags(&ctx->pin_in_done, cudaEventDisableTiming));
    QB_CUDA(cudaEventCreateWithFlags(&ctx->pin_entries_done, cudaEventDisableTiming));
#define QB_CONFIGURE(R_, K_)                                                                                            \
    QB_TRY(configure_kernel(qb::sweep_kernel<double, R_, K_, uint32_t>, qb::sweep_smem_bytes<double, R_, K_>())); \
    QB_TRY(configure_kernel(qb::sweep_kernel<float, R_, K_, uint32_t>, qb::sweep_smem_bytes<float, R_, K_>()));   \
    QB_TRY(configure_kernel(qb::sweep_kernel<double, R_, K_, uint64_t>, qb::sweep_smem_bytes<double, R_, K_>())); \
    QB_TRY(configure_kernel(qb::sweep_kernel<float, R_, K_, uint64_t>, qb::sweep_smem_bytes<float, R_, K_>()));
    QB_CONFIGURE(4, 11)
    QB_CONFIGURE(4, 12)
    QB_CONFIGURE(3, 11)
#undef QB_CONFIGURE
    if (const char* e = std::getenv("QB_TILES_LOG2")) ctx->tiles_log2 = std::max(0, std::atoi(e));
    if (const char* e = std::getenv("QB_SWEEP_STREAMS")) ctx->sweep_streams = std::min(8, std::max(1, std::atoi(e)));
    if (const char* e = std::getenv("QB_SWEEP_GROUP")) ctx->sweep_group = std::max(0, std::atoi(e));
    if (const char* e = std::getenv("QB_GRAPHS")) ctx->use_graphs = std::atoi(e) != 0;
    if (const char* e = std::getenv("QB_PDL")) ctx->pdl = std::max(0, std::atoi(e));
    if (const char* e = std::getenv("QB_ZERO_COPY")) ctx->zero_copy = std::atoi(e) != 0;
    if (const char* e = std::getenv("QB_L2_PREFETCH")) ctx->l2_prefetch = std::atoi(e) ? 1 : 0;
    QB_CUDA(cudaEventCreateWithFlags(&ctx->fork_event, cudaEventDisableTiming));
    for (int i = 0; i < 8; ++i) {
        QB_CUDA(cudaStreamCreateWithFlags(&ctx->aux_streams[i], cudaStreamNonBlocking));
        QB_CUDA(cudaEventCreateWithFlags(&ctx->join_events[i], cudaEventDisableTiming));
    }
    *out = ctx.release();
    return QB_OK;
}

int qb_context_destroy(qb_context* ctx) {
    if (!ctx) return QB_OK;
    ctx->worker.reset();  // stops and joins the context's host thread
    DeviceScope scope(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    ctx->single_graphs.clear();
    ctx->batches.clear();
    ctx->plans.clear();
    ctx->hams.clear();
    ctx->observables.clear();
    ctx->pin_in.release(), ctx->pin_out.release(), ctx->scratch.release();
    if (ctx->pin_in_done) cudaEventDestroy(ctx->pin_in_done);
    if (ctx->pin_entries_done) cudaEventDestroy(ctx->pin_entries_done);
    if (ctx->fork_event) cudaEventDestroy(ctx->fork_event);
    for (int i = 0; i < 8; ++i) {
        if (ctx->join_events[i]) cudaEventDestroy(ctx->join_events[i]);
        if (ctx->aux_streams[i]) cudaStreamDestroy(ctx->aux_streams[i]);
    }
    ctx->pin_entries.release();
    ctx->pin_res.release();
    if (ctx->owns_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return QB_OK;
}

void* qb_context_stream(qb_context* ctx) { return ctx ? static_cast<void*>(ctx->stream) : nullptr; }

int64_t qb_context_launch_count(qb_context* ctx) { return ctx ? ctx->launches : 0; }

int qb_context_set_workspace_limit(qb_context* ctx, uint64_t bytes) {
    if (!ctx) return fail(QB_ERR_INVALID, "null context");
    ctx->workspace_limit = bytes;
    return QB_OK;
}

int qb_context_set_index_width(qb_context* ctx, int bits) {
    if (!ctx) return fail(QB_ERR_INVALID, "null context");
    if (bits != 32 && bits != 64) return fail(QB_ERR_INVALID, "index width must be 32 (automatic) or 64");
    std::lock_guard<std::mutex> lock(ctx->mu);
    ctx->force_idx64 = bits == 64;
    return QB_OK;
}

int qb_context_synchronize(qb_context* ctx) {
    if (!ctx) return fail(QB_ERR_INVALID, "null context");
    QB_ON_DEVICE(ctx);
    QB_CUDA(cudaStreamSynchronize(ctx->stream));
    return QB_OK;
}

// ---- plans ------------------------------------------------------------------------------------------
int qb_plan_create(qb_context* ctx, int n_qubits, int dtype, int tile_bits, int reg_bits, int n_params, int n_ops, const qb_op_angles* ops, int n_sweeps,
                   const qb_sweep* sweeps, int n_passes, const qb_pass* passes, int n_pass_ops, const qb_pass_op* pass_ops,
                   const int32_t* init_ops, int64_t* plan_id) {
    if (!ctx || !plan_id) return fail(QB_ERR_INVALID, "null argument");
    if (n_qubits < 1 || n_qubits > 40) return fail(QB_ERR_INVALID, "n_qubits out of range");
    if (dtype != QB_C128 && dtype != QB_C64) return fail(QB_ERR_INVALID, "dtype must be QB_C128 or QB_C64");
    if (n_sweeps < 1 || n_passes < 1) return fail(QB_ERR_INVALID, "a plan needs at least one sweep with one pass");
    if (reg_bits != QB_REG_BITS && !(reg_bits == 3 && tile_bits == 11)) return fail(QB_ERR_INVALID, "reg_bits must be 4 (or 3 with 2^11 tiles)");
    const int thread_bits = tile_bits - reg_bits;
    if (tile_bits != 11 && tile_bits != 12) return fail(QB_ERR_INVALID, "tile_bits must be 11 or 12");
    const int n_eff = std::max(n_qubits, tile_bits);
    // validate the program: everything the kernel indexes with must be in range
    for (int s = 0; s < n_sweeps; ++s) {
        const qb_sweep& sw = sweeps[s];
        if (sw.pass_begin < 0 || sw.pass_end > n_passes || sw.pass_end <= sw.pass_begin)
            return fail(QB_ERR_INVALID, "sweep " + std::to_string(s) + ": bad pass range");
        if (sw.pass_end - sw.pass_begin > qb::kMaxSweepPasses) return fail(QB_ERR_INVALID, "sweep has too many passes");
        uint64_t mask = 0;
        for (int i = 0; i < tile_bits; ++i) {
            const int q = sw.tile_qubits[i];
            if (q < 0 || q >= n_eff || ((mask >> q) & 1)) return fail(QB_ERR_INVALID, "sweep " + std::to_string(s) + ": bad tile qubit");
            if (i && q <= sw.tile_qubits[i - 1]) return fail(QB_ERR_INVALID, "tile qubits must ascend");
            mask |= 1ull << q;
        }
        const int ob = passes[sw.pass_begin].op_begin, oe = passes[sw.pass_end - 1].op_end;
        if (sw.op_begin != ob || sw.op_end != oe) return fail(QB_ERR_INVALID, "sweep op range does not match its passes");
        if (ob < 0 || oe > n_pass_ops || oe < ob || oe - ob > qb::kMaxSweepOps)
            return fail(QB_ERR_INVALID, "sweep " + std::to_string(s) + ": bad op range / too many ops");
        for (int p = sw.pass_begin; p < sw.pass_end; ++p) {
            const qb_pass& ps = passes[p];
            uint32_t used = 0;
            for (int i = 0; i < reg_bits; ++i) {
                const int b = ps.reg_bits[i];
                if (b < 0 || b >= tile_bits || ((used >> b) & 1)) return fail(QB_ERR_INVALID, "bad register bit");
                used |= 1u << b;
            }
            for (int i = 0; i < thread_bits; ++i) {
                const int b = ps.thread_bits[i];
                if (b >= tile_bits || ((used >> b) & 1)) return fail(QB_ERR_INVALID, "bad thread bit");
                used |= 1u << b;
            }
            if (p > sw.pass_begin && ps.op_begin != passes[p - 1].op_end) return fail(QB_ERR_INVALID, "pass op ranges must be contiguous");
            if (ps.flags & QB_PASS_WARP_LOCAL) {  // claim must hold: same tile bits on the warp-index bits of the next pass
                if (p + 1 >= sw.pass_end) return fail(QB_ERR_INVALID, "warp-local flag on the last pass of a sweep");
                for (int i = 5; i < thread_bits; ++i)
                    if (ps.thread_bits[i] != passes[p + 1].thread_bits[i]) return fail(QB_ERR_INVALID, "warp-local exchange with different warp bits");
            }
            for (int o = ps.op_begin; o < ps.op_end; ++o) {
                const qb_pass_op& po = pass_ops[o];
                if (po.op_index < 0 || po.op_index >= n_ops) return fail(QB_ERR_INVALID, "op index out of range");
                if (po.kind == QB_OP_DENSE && (po.tgt_kind != QB_K_REG || po.tgt_pos >= reg_bits))
                    return fail(QB_ERR_INVALID, "dense op target must be a register bit");
                auto bad = [&](int kind, int pos) {
                    if (kind == QB_K_REG) return pos >= reg_bits;
                    if (kind == QB_K_THREAD) return pos >= tile_bits;
                    if (kind == QB_K_EXT) return pos >= 64;
                    return kind != QB_K_NONE;
                };
                if (bad(po.tgt_kind, po.tgt_pos) || po.tgt_kind == QB_K_NONE || bad(po.ctrl_kind, po.ctrl_pos))
                    return fail(QB_ERR_INVALID, "bad operand kind/position");
                // the pre-decoded dispatch fields must agree with the descriptive ones
                auto gq = [&](int kind, int pos) { return kind == QB_K_THREAD ? sw.tile_qubits[pos] : (kind == QB_K_EXT ? pos : 0xFF); };
                const int cb = po.ctrl_kind == QB_K_REG ? int(po.ctrl_pos) : -1;
                int variant, tq = 0xFF;
                if (po.kind == QB_OP_DENSE) variant = 6 * po.tgt_pos + cb + 1;
                else if (cb >= 0) variant = 40, tq = gq(po.tgt_kind, po.tgt_pos);
                else if (po.tgt_kind == QB_K_REG) variant = 33 + po.tgt_pos;
                else variant = 32, tq = gq(po.tgt_kind, po.tgt_pos);
                if (po.kind == QB_OP_DENSE && cb == int(po.tgt_pos)) return fail(QB_ERR_INVALID, "control equals target");
                if (po.variant != variant || po.ctrl_qubit != gq(po.ctrl_kind, po.ctrl_pos) || po.tgt_qubit != tq)
                    return fail(QB_ERR_INVALID, "pre-decoded dispatch fields are inconsistent");
            }
        }
    }
    for (int o = 0; o < n_ops; ++o)
        for (int j = 0; j < 4; ++j)
            if (ops[o].slot[j] >= n_params || ops[o].slot2[j] >= n_params) return fail(QB_ERR_INVALID, "angle slot out of range");
    bool has_init = false;
    if (init_ops) {
        std::vector<char> used(size_t(std::max(n_ops, 1)), 0);
        for (int q = 0; q < n_eff; ++q) {
            if (init_ops[q] < 0) continue;
            if (init_ops[q] >= n_ops || used[init_ops[q]]) return fail(QB_ERR_INVALID, "bad init op index");
            used[init_ops[q]] = 1;
            has_init = true;
        }
        for (int o = 0; o < n_pass_ops; ++o)
            if (used[pass_ops[o].op_index]) return fail(QB_ERR_INVALID, "an init op also appears in a pass");
    }

    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    auto pl = std::make_unique<Plan>();
    pl->n_qubits = n_qubits, pl->n_eff = n_eff, pl->dtype = dtype, pl->tile_bits = tile_bits, pl->reg_bits = reg_bits, pl->n_params = n_params, pl->n_ops = n_ops, pl->n_sweeps = n_sweeps, pl->n_pass_ops = n_pass_ops;
    QB_TRY(upload(ctx, pl->sweeps, sweeps, sizeof(qb_sweep) * size_t(n_sweeps)));
    QB_TRY(upload(ctx, pl->passes, passes, sizeof(qb_pass) * size_t(n_passes)));
    QB_TRY(upload(ctx, pl->pass_ops, pass_ops, sizeof(qb_pass_op) * size_t(n_pass_ops)));
    QB_TRY(upload(ctx, pl->angles, ops, sizeof(qb_op_angles) * size_t(n_ops)));
    pl->has_init = has_init;
    if (has_init) QB_TRY(upload(ctx, pl->init_ops, init_ops, sizeof(int32_t) * size_t(n_eff)));
    QB_CUDA(cudaStreamSynchronize(ctx->stream));
    *plan_id = ctx->next_id++;
    ctx->plans[*plan_id] = std::move(pl);
    return QB_OK;
}

int qb_plan_set_prefix(qb_context* ctx, int64_t plan_id, int64_t prefix_plan_id) {
    if (!ctx) return fail(QB_ERR_INVALID, "null context");
    std::lock_guard<std::mutex> lock(ctx->mu);
    Plan* pl = find_plan(ctx, plan_id);
    Plan* pre = find_plan(ctx, prefix_plan_id);
    if (!pl || !pre) return fail(QB_ERR_NOT_FOUND, "unknown plan id");
    if (pl->has_init) return fail(QB_ERR_INVALID, "a prefixed plan must be compiled for application to an existing state");
    if (pre->n_params != 0 || pre->prefix_id || pre->n_eff != pl->n_eff || pre->dtype != pl->dtype || pre->n_qubits != pl->n_qubits)
        return fail(QB_ERR_INVALID, "prefix plan must be parameter-free, un-prefixed and of the same shape");
    QB_ON_DEVICE(ctx);
    cudaStreamSynchronize(ctx->stream);
    drop_single_graphs(ctx, plan_id, 0);  // a cached graph of this plan starts it from |0...0>, not from the prefix state
    pl->prefix_id = prefix_plan_id;
    pl->prefix_ready = false;
    ctx->epoch++;  // assembled batches may hold this plan's old start
    return QB_OK;
}

int qb_plan_destroy(qb_context* ctx, int64_t plan_id) {
    if (!ctx) return fail(QB_ERR_INVALID, "null context");
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    cudaStreamSynchronize(ctx->stream);
    drop_single_graphs(ctx, plan_id, 0);
    ctx->epoch++;
    return ctx->plans.erase(plan_id) ? QB_OK : fail(QB_ERR_NOT_FOUND, "unknown plan id");
}

// ---- Hamiltonians -------------------------------------------------------------------------------------
int qb_hamiltonian_create(qb_context* ctx, int n_qubits, int n_terms, const uint64_t* x_masks, const uint64_t* z_masks,
                          const double* coeff_re, const double* coeff_im, int build_table, int64_t* ham_id) {
    if (!ctx || !ham_id) return fail(QB_ERR_INVALID, "null argument");
    if (n_qubits < 1 || n_qubits > 40 || n_terms < 0) return fail(QB_ERR_INVALID, "bad Hamiltonian shape");
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    auto ham = std::make_unique<Ham>();
    ham->n_qubits = n_qubits;
    // group by x mask, keeping first-appearance order; weights w = coeff * i^{#Y}
    std::vector<uint64_t> xs;
    std::vector<std::vector<int>> members;
    QB_TRY(group_by_xmask(n_qubits, n_terms, x_masks, z_masks, xs, members));
    std::vector<uint64_t> dz;
    std::vector<double> dc;
    for (size_t g = 0; g < xs.size(); ++g) {
        std::vector<uint64_t> z;
        std::vector<double> wr, wi;
        for (int t : members[g]) {
            const int ny = __builtin_popcountll(x_masks[t] & z_masks[t]) & 3;
            const double re = coeff_re[t], im = coeff_im ? coeff_im[t] : 0.0;
            double r = re, i = im;  // multiply by i^ny
            if (ny == 1) r = -im, i = re;
            else if (ny == 2) r = -re, i = -im;
            else if (ny == 3) r = im, i = -re;
            z.push_back(z_masks[t]), wr.push_back(r), wi.push_back(i);
            if (xs[g] == 0) dz.push_back(z_masks[t]), dc.push_back(re);
        }
        if (xs[g] != 0) ham->diagonal = false;
        auto grp = std::make_unique<Group>();
        grp->xmask = xs[g];
        grp->n_terms = int(z.size());
        QB_TRY(upload(ctx, grp->z, z.data(), sizeof(uint64_t) * z.size()));
        QB_TRY(upload(ctx, grp->wr, wr.data(), sizeof(double) * wr.size()));
        QB_TRY(upload(ctx, grp->wi, wi.data(), sizeof(double) * wi.size()));
        QB_CUDA(cudaStreamSynchronize(ctx->stream));
        if (xs[g] == 0) ham->groups.insert(ham->groups.begin(), std::move(grp));
        else ham->groups.push_back(std::move(grp));
    }
    ham->n_diag = int(dz.size());
    QB_TRY(upload(ctx, ham->diag_z, dz.data(), sizeof(uint64_t) * dz.size()));
    QB_TRY(upload(ctx, ham->diag_c, dc.data(), sizeof(double) * dc.size()));
    QB_CUDA(cudaStreamSynchronize(ctx->stream));
    if (build_table && ham->n_diag > 0) {
        const int n_eff = std::max(n_qubits, QB_TILE_BITS);
        QB_TRY(ham->table.reserve(sizeof(double) * (uint64_t(1) << n_eff)));
        ham->table_n_eff = n_eff;
        QB_TRY(fill_diag_table(ctx, *ham, ham->table.as<double>(), n_eff));
        QB_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    {   // schedule the non-diagonal x-mask groups into tile sweeps
        const int n_eff = std::max(n_qubits, qb::kExpTileBits);
        ham->tile_n_eff = n_eff;
        std::vector<uint64_t> gx(ham->groups.size());
        std::vector<int> pending;
        for (size_t g = 0; g < ham->groups.size(); ++g) {
            gx[g] = ham->groups[g]->xmask;
            if (gx[g] != 0) pending.push_back(int(g));
        }
        TilePlan tp = plan_tile_sweeps(n_eff, gx, pending);
        ham->tile_sweeps = tp.sweeps, ham->tile_sweep_groups = tp.sweep_groups, ham->generic_groups = tp.generic;
        std::vector<qb::ExpTileGroup> tgroups;
        std::vector<uint64_t> tz;
        std::vector<double> twr, twi;
        std::vector<std::vector<uint64_t>> host_z(ham->groups.size());
        std::vector<std::vector<double>> host_wr(ham->groups.size()), host_wi(ham->groups.size());
        for (size_t g = 0; g < xs.size(); ++g) {  // recover host copies of the per-group terms (same order as uploaded)
            size_t slot = 0;
            for (; slot < ham->groups.size(); ++slot)
                if (ham->groups[slot]->xmask == xs[g]) break;
            for (int t : members[g]) {
                const int ny = __builtin_popcountll(x_masks[t] & z_masks[t]) & 3;
                const double re = coeff_re[t], im = coeff_im ? coeff_im[t] : 0.0;
                double r = re, i = im;
                if (ny == 1) r = -im, i = re;
                else if (ny == 2) r = -re, i = -im;
                else if (ny == 3) r = im, i = -re;
                host_z[slot].push_back(z_masks[t]), host_wr[slot].push_back(r), host_wi[slot].push_back(i);
            }
        }
        for (const auto& chosen : tp.sweep_groups)
            for (int g : chosen) {
                qb::ExpTileGroup tg{};
                tg.xloc = tp.xloc[g];
                tg.term_begin = int(tz.size());
                tz.insert(tz.end(), host_z[g].begin(), host_z[g].end());
                twr.insert(twr.end(), host_wr[g].begin(), host_wr[g].end());
                twi.insert(twi.end(), host_wi[g].begin(), host_wi[g].end());
                tg.term_end = int(tz.size());
                tg.trivial = (host_z[g].size() == 1 && host_z[g][0] == 0) ? 1 : 0;
                tgroups.push_back(tg);
            }
        if (!tgroups.empty()) {
            QB_TRY(upload(ctx, ham->tile_groups, tgroups.data(), sizeof(qb::ExpTileGroup) * tgroups.size()));
            QB_TRY(upload(ctx, ham->tile_z, tz.data(), sizeof(uint64_t) * tz.size()));
            QB_TRY(upload(ctx, ham->tile_wr, twr.data(), sizeof(double) * twr.size()));
            QB_TRY(upload(ctx, ham->tile_wi, twi.data(), sizeof(double) * twi.size()));
            QB_CUDA(cudaStreamSynchronize(ctx->stream));
        }
    }
    *ham_id = ctx->next_id++;
    ctx->hams[*ham_id] = std::move(ham);
    return QB_OK;
}

int qb_hamiltonian_destroy(qb_context* ctx, int64_t ham_id) {
    if (!ctx) return fail(QB_ERR_INVALID, "null context");
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    cudaStreamSynchronize(ctx->stream);
    drop_single_graphs(ctx, 0, ham_id);
    ctx->epoch++;
    return ctx->hams.erase(ham_id) ? QB_OK : fail(QB_ERR_NOT_FOUND, "unknown Hamiltonian id");
}

int qb_hamiltonian_diag_energies(qb_context* ctx, int64_t ham_id, int64_t n_states, const uint64_t* states, double* out_energies) {
    if (!ctx || (n_states > 0 && (!states || !out_energies))) return fail(QB_ERR_INVALID, "null argument");
    if (n_states <= 0) return QB_OK;
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    Ham* ham = find_ham(ctx, ham_id);
    if (!ham) return fail(QB_ERR_NOT_FOUND, "unknown Hamiltonian id");
    if (!ham->diagonal) return fail(QB_ERR_INVALID, "Hamiltonian has non-diagonal terms");
    const size_t bytes = sizeof(uint64_t) * size_t(n_states);
    QB_TRY(ctx->scratch.reserve(2 * bytes));
    QB_CUDA(cudaEventSynchronize(ctx->pin_in_done));
    QB_TRY(ctx->pin_in.reserve(bytes));
    QB_TRY(ctx->pin_out.reserve(bytes));
    std::memcpy(ctx->pin_in.p, states, bytes);
    uint64_t* d_states = ctx->scratch.as<uint64_t>();
    double* d_out = reinterpret_cast<double*>(d_states + n_states);
    QB_CUDA(cudaMemcpyAsync(d_states, ctx->pin_in.p, bytes, cudaMemcpyHostToDevice, ctx->stream));
    const int blocks = int(std::min<int64_t>(1024, (n_states + 255) / 256));
    qb::diag_lookup_kernel<<<blocks, 256, 0, ctx->stream>>>(d_states, n_states, ham->diag_z.as<uint64_t>(), ham->diag_c.as<double>(),
                                                            ham->n_diag, d_out);
    QB_TRY(check_launch(ctx, "diag_lookup_kernel"));
    QB_CUDA(cudaMemcpyAsync(ctx->pin_out.p, d_out, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    QB_CUDA(cudaStreamSynchronize(ctx->stream));
    std::memcpy(out_energies, ctx->pin_out.p, bytes);
    return QB_OK;
}

// ---- observable sets ----------------------------------------------------------------------------------
int qb_observables_create(qb_context* ctx, int n_qubits, int n_obs, const int64_t* term_offsets, const uint64_t* x_masks,
                          const uint64_t* z_masks, const double* coeff_re, const double* coeff_im, int64_t* obs_id) {
    (void)coeff_im;  // every string is Hermitian, <P_t> is real: Re(c <P_t>) = Re(c) <P_t>
    if (!ctx || !term_offsets || !obs_id) return fail(QB_ERR_INVALID, "null argument");
    if (n_qubits < 1 || n_qubits > 40) return fail(QB_ERR_INVALID, "bad observable width");
    if (n_obs < 1) return fail(QB_ERR_INVALID, "an observable set needs at least one observable");
    if (term_offsets[0] != 0) return fail(QB_ERR_INVALID, "term_offsets[0] must be 0");
    for (int j = 0; j < n_obs; ++j)
        if (term_offsets[j + 1] < term_offsets[j]) return fail(QB_ERR_INVALID, "term_offsets must not decrease");
    const int64_t total = term_offsets[n_obs];
    if (total > (int64_t(1) << 30)) return fail(QB_ERR_INVALID, "too many terms");
    if (total > 0 && (!x_masks || !z_masks || !coeff_re)) return fail(QB_ERR_INVALID, "null argument");
    // union of the distinct (x, z) strings in first-appearance order; CSR rows over union indices, duplicates summed
    std::map<std::pair<uint64_t, uint64_t>, int> index_of;
    std::vector<uint64_t> ux, uz;
    std::vector<int64_t> row_begin(size_t(n_obs) + 1, 0);
    std::vector<int32_t> cols;
    std::vector<double> coeff;
    for (int j = 0; j < n_obs; ++j) {
        std::map<int, double> row;  // union index -> coefficient (ascending term order)
        for (int64_t t = term_offsets[j]; t < term_offsets[j + 1]; ++t) {
            if ((x_masks[t] | z_masks[t]) >> n_qubits) return fail(QB_ERR_INVALID, "Pauli term acts outside the register");
            auto ins = index_of.emplace(std::make_pair(x_masks[t], z_masks[t]), int(ux.size()));
            if (ins.second) ux.push_back(x_masks[t]), uz.push_back(z_masks[t]);
            row[ins.first->second] += coeff_re[t];
        }
        for (const auto& e : row) cols.push_back(e.first), coeff.push_back(e.second);
        row_begin[j + 1] = int64_t(cols.size());
    }
    auto ob = std::make_unique<Obs>();
    ob->n_qubits = n_qubits, ob->n_obs = n_obs, ob->n_terms = int(ux.size());
    ob->n_eff = std::max(n_qubits, qb::kExpTileBits);
    std::vector<uint64_t> xs;
    std::vector<std::vector<int>> members;
    QB_TRY(group_by_xmask(n_qubits, ob->n_terms, ux.data(), uz.data(), xs, members));
    std::vector<int> pending(xs.size());
    std::iota(pending.begin(), pending.end(), 0);
    for (size_t g = 0; g < xs.size(); ++g)  // the diagonal group (|psi_k|^2, no partner) first
        if (xs[g] == 0) std::rotate(pending.begin(), pending.begin() + g, pending.begin() + g + 1);
    const TilePlan tp = plan_tile_sweeps(ob->n_eff, xs, pending);
    // device order of the strings: sweep after sweep, group after group, then the generic groups
    std::vector<int> slot_of(ux.size());
    std::vector<uint64_t> dz;
    std::vector<int8_t> dim;
    std::vector<double> dsign;
    std::vector<qb::TermGroup> records;
    auto place = [&](int g) {
        qb::TermGroup rec{};
        rec.xmask = xs[g], rec.xloc = tp.xloc[g], rec.term_begin = int(dz.size()), rec.real_only = 1;
        for (int u : members[g]) {
            const int ny = __builtin_popcountll(ux[u] & uz[u]) & 3;
            slot_of[u] = int(dz.size());
            dz.push_back(uz[u]), dim.push_back(int8_t(ny & 1)), dsign.push_back((ny == 1 || ny == 2) ? -1.0 : 1.0);
            if (ny & 1) rec.real_only = 0;
        }
        rec.term_end = int(dz.size());
        return rec;
    };
    ob->tile_sweeps = tp.sweeps;
    for (const auto& chosen : tp.sweep_groups) {
        const int first = int(dz.size());
        for (int g : chosen) records.push_back(place(g));
        ob->sweep_terms.emplace_back(first, int(dz.size()));
    }
    for (int g : tp.generic) ob->generic.push_back(place(g));
    for (auto& c : cols) c = slot_of[c];
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    QB_TRY(upload(ctx, ob->groups, records.data(), sizeof(qb::TermGroup) * records.size()));
    QB_TRY(upload(ctx, ob->z, dz.data(), sizeof(uint64_t) * dz.size()));
    QB_TRY(upload(ctx, ob->im, dim.data(), dim.size()));
    QB_TRY(upload(ctx, ob->sign, dsign.data(), sizeof(double) * dsign.size()));
    QB_TRY(upload(ctx, ob->row_begin, row_begin.data(), sizeof(int64_t) * row_begin.size()));
    QB_TRY(upload(ctx, ob->cols, cols.data(), sizeof(int32_t) * cols.size()));
    QB_TRY(upload(ctx, ob->coeff, coeff.data(), sizeof(double) * coeff.size()));
    QB_CUDA(cudaStreamSynchronize(ctx->stream));
    *obs_id = ctx->next_id++;
    ctx->observables[*obs_id] = std::move(ob);
    return QB_OK;
}

int qb_observables_destroy(qb_context* ctx, int64_t obs_id) {
    if (!ctx) return fail(QB_ERR_INVALID, "null context");
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    cudaStreamSynchronize(ctx->stream);
    return ctx->observables.erase(obs_id) ? QB_OK : fail(QB_ERR_NOT_FOUND, "unknown observable set id");
}

// ---- resident batches -----------------------------------------------------------------------------------
int qb_batch_create(qb_context* ctx, int batch, const int64_t* plan_ids, int64_t ham_id, int64_t* batch_id) {
    if (!ctx || !plan_ids || !batch_id) return fail(QB_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    Ham* ham = nullptr;
    if (ham_id) {
        ham = find_ham(ctx, ham_id);
        if (!ham) return fail(QB_ERR_NOT_FOUND, "unknown Hamiltonian id");
    }
    auto b = std::make_unique<DeviceBatch>();
    b->ham_id = ham_id;
    QB_TRY(build_batch(ctx, *b, batch, plan_ids, ham, nullptr, 1, 0));
    *batch_id = ctx->next_id++;
    ctx->batches[*batch_id] = std::move(b);
    return QB_OK;
}

static DeviceBatch* find_batch(qb_context* ctx, int64_t id) {
    auto it = ctx->batches.find(id);
    return it == ctx->batches.end() ? nullptr : it->second.get();
}

// The resident batch `id`, re-assembled first when a plan or Hamiltonian was destroyed or a plan given a prefix since it was
// built (its entries may point into freed device memory or miss the new start): QB_ERR_NOT_FOUND, before anything is launched,
// when one of its plans or its Hamiltonian is gone.  The parameter layout depends on the plans alone, so uploaded parameters
// stay valid across a re-assembly.
static int current_batch(qb_context* ctx, int64_t id, DeviceBatch** out) {
    DeviceBatch* b = find_batch(ctx, id);
    if (!b) return fail(QB_ERR_NOT_FOUND, "unknown batch id");
    if (b->built_epoch != ctx->epoch) {
        const Ham* ham = nullptr;
        if (b->ham_id && !(ham = find_ham(ctx, b->ham_id)))
            return fail(QB_ERR_NOT_FOUND, "Hamiltonian " + std::to_string(b->ham_id) + " of the batch no longer exists");
        const std::vector<int64_t> ids = b->built_ids;  // (build_batch clears built_ids before it reads the list)
        const int rc = build_batch(ctx, *b, int(ids.size()), ids.data(), ham, nullptr, 1, 0);
        if (rc != QB_OK) {
            b->built_ids = ids;  // still stale (built_epoch is unchanged): the next call tries again and fails the same way
            return rc;
        }
    }
    *out = b;
    return QB_OK;
}

int qb_batch_set_params(qb_context* ctx, int64_t batch_id, const double* params, const int64_t* param_offsets) {
    if (!ctx || !param_offsets) return fail(QB_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    DeviceBatch* b = nullptr;
    QB_TRY(current_batch(ctx, batch_id, &b));
    return batch_upload_params(ctx, *b, params, param_offsets);
}

int qb_batch_run(qb_context* ctx, int64_t batch_id) {
    if (!ctx) return fail(QB_ERR_INVALID, "null context");
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    DeviceBatch* b = nullptr;
    QB_TRY(current_batch(ctx, batch_id, &b));
    const int64_t before = ctx->launches;
    QB_TRY(launch_circuits(ctx, *b, nullptr));
    if (b->ham) QB_TRY(launch_expectation(ctx, *b));
    b->launches_per_run = ctx->launches - before;
    return QB_OK;
}

int qb_batch_run_timed(qb_context* ctx, int64_t batch_id, int max_launches, float* sweep_ms, int32_t* sweep_states, int* n_launches) {
    if (!ctx || !sweep_ms || !sweep_states || !n_launches) return fail(QB_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    DeviceBatch* b = nullptr;
    QB_TRY(current_batch(ctx, batch_id, &b));
    if (max_launches < b->max_sweeps) return fail(QB_ERR_INVALID, "output arrays too small");
    std::vector<cudaEvent_t> events(2 * size_t(b->max_sweeps));
    for (auto& e : events) QB_CUDA(cudaEventCreate(&e));
    int rc = launch_circuits(ctx, *b, events.data());
    if (rc == QB_OK && b->ham) rc = launch_expectation(ctx, *b);
    cudaError_t se = cudaStreamSynchronize(ctx->stream);
    if (rc == QB_OK && se == cudaSuccess) {
        for (int s = 0; s < b->max_sweeps; ++s) {
            cudaEventElapsedTime(&sweep_ms[s], events[2 * s], events[2 * s + 1]);
            sweep_states[s] = b->active[s];
        }
        *n_launches = b->max_sweeps;
    }
    for (auto& e : events) cudaEventDestroy(e);
    if (rc != QB_OK) return rc;
    if (se != cudaSuccess) return fail(QB_ERR_CUDA, std::string("cudaStreamSynchronize: ") + cudaGetErrorString(se));
    return QB_OK;
}

int qb_batch_read(qb_context* ctx, int64_t batch_id, double* out_values) {
    if (!ctx || !out_values) return fail(QB_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    DeviceBatch* b = nullptr;
    QB_TRY(current_batch(ctx, batch_id, &b));
    return batch_read(ctx, *b, out_values);
}

int qb_batch_destroy(qb_context* ctx, int64_t batch_id) {
    if (!ctx) return fail(QB_ERR_INVALID, "null context");
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    cudaStreamSynchronize(ctx->stream);
    return ctx->batches.erase(batch_id) ? QB_OK : fail(QB_ERR_NOT_FOUND, "unknown batch id");
}

int qb_batch_stats(qb_context* ctx, int64_t batch_id, int64_t* n_sweep_launches, int64_t* n_state_sweeps, int64_t* sweep_bytes,
                   int64_t* n_kernel_launches) {
    if (!ctx) return fail(QB_ERR_INVALID, "null context");
    std::lock_guard<std::mutex> lock(ctx->mu);
    DeviceBatch* b = find_batch(ctx, batch_id);
    if (!b) return fail(QB_ERR_NOT_FOUND, "unknown batch id");
    if (n_sweep_launches) *n_sweep_launches = b->max_sweeps;
    if (n_state_sweeps) *n_state_sweeps = b->n_state_sweeps;
    if (sweep_bytes) *sweep_bytes = int64_t(2 * amp_bytes(b->dtype)) << b->n_eff;
    if (n_kernel_launches) *n_kernel_launches = b->launches_per_run;
    return QB_OK;
}

// ---- one-shot batched evaluation ---------------------------------------------------------------------
int qb_evaluate_expectation(qb_context* ctx, int batch, const int64_t* plan_ids, const double* params, const int64_t* param_offsets,
                            int64_t ham_id, double* out_values) {
    if (!ctx || !plan_ids || !param_offsets || !out_values) return fail(QB_ERR_INVALID, "null argument");
    if (batch <= 0) return QB_OK;
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    Ham* ham = find_ham(ctx, ham_id);
    if (!ham) return fail(QB_ERR_NOT_FOUND, "unknown Hamiltonian id");
    Plan* first = find_plan(ctx, plan_ids[0]);
    if (!first) return fail(QB_ERR_NOT_FOUND, "unknown plan id " + std::to_string(plan_ids[0]));
    if (batch <= kMaxGraphCopies && std::all_of(plan_ids, plan_ids + batch, [&](int64_t id) { return id == plan_ids[0]; })) {
        // the optimizer loop's call (one circuit, one or a few parameter points): replay the evaluation's CUDA graph
        bool handled = false;
        QB_TRY(evaluate_single_graph(ctx, plan_ids[0], first, ham, ham_id, batch, params, param_offsets, out_values, &handled));
        if (handled) return QB_OK;
    }
    const int chunk = int(std::min<size_t>(size_t(batch), max_batch_for(ctx, first)));
    return run_oneshot(ctx, batch, plan_ids, params, param_offsets, ham, chunk, [&](DeviceBatch& b, int lo) {
        QB_TRY(launch_expectation(ctx, b));
        return batch_read(ctx, b, out_values + lo);
    });
}

int qb_sample(qb_context* ctx, int batch, const int64_t* plan_ids, const double* params, const int64_t* param_offsets, int shots,
              const double* uniforms, int64_t* out_indices) {
    if (!ctx || !plan_ids || !param_offsets || !uniforms || !out_indices) return fail(QB_ERR_INVALID, "null argument");
    if (batch <= 0 || shots <= 0) return QB_OK;
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    Plan* first = find_plan(ctx, plan_ids[0]);
    if (!first) return fail(QB_ERR_NOT_FOUND, "unknown plan id " + std::to_string(plan_ids[0]));
    const int chunk = int(std::min<size_t>(size_t(batch), max_batch_for(ctx, first)));
    return run_oneshot(ctx, batch, plan_ids, params, param_offsets, nullptr, chunk, [&](DeviceBatch& b, int lo) {
        const int n = b.batch;
        const uint64_t size = uint64_t(1) << b.n_eff;
        const uint64_t n_chunks = size >> qb::kChunkBits;
        const size_t u_bytes = sizeof(double) * size_t(n) * size_t(shots);
        const size_t c_bytes = sizeof(double) * size_t(n) * n_chunks;
        QB_TRY(ctx->scratch.reserve(2 * u_bytes + c_bytes));
        double* d_uniforms = ctx->scratch.as<double>();
        int64_t* d_indices = reinterpret_cast<int64_t*>(d_uniforms + size_t(n) * shots);
        double* d_chunks = reinterpret_cast<double*>(d_indices + size_t(n) * shots);
        QB_CUDA(cudaEventSynchronize(ctx->pin_in_done));
        QB_TRY(ctx->pin_in.reserve(u_bytes));
        QB_TRY(ctx->pin_out.reserve(u_bytes));
        // uniforms in sorted (device) order
        double* stage = static_cast<double*>(ctx->pin_in.p);
        gather_rows(stage, uniforms + size_t(lo) * shots, b.order, sizeof(double) * size_t(shots));
        QB_CUDA(cudaMemcpyAsync(d_uniforms, stage, u_bytes, cudaMemcpyHostToDevice, ctx->stream));
        QB_TRY(with_dtype(b.dtype, [&](auto t) {
            using T = decltype(t);
            return launch_sampling_t<T>(ctx, b.states.as<typename qb::Cx<T>::type>(), size, n, uint64_t(1) << b.n_qubits, d_uniforms, shots, d_chunks,
                                        d_indices);
        }));
        QB_CUDA(cudaMemcpyAsync(ctx->pin_out.p, d_indices, u_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        QB_CUDA(cudaStreamSynchronize(ctx->stream));
        scatter_rows(out_indices + size_t(lo) * shots, ctx->pin_out.p, b.order, sizeof(int64_t) * size_t(shots));
        return QB_OK;
    });
}

int qb_evaluate_cvar(qb_context* ctx, int batch, const int64_t* plan_ids, const double* params, const int64_t* param_offsets,
                     int64_t ham_id, double alpha, double* out_values) {
    if (!ctx || !plan_ids || !param_offsets || !out_values) return fail(QB_ERR_INVALID, "null argument");
    if (!(alpha > 0.0 && alpha <= 1.0)) return fail(QB_ERR_INVALID, "alpha must be in the range (0, 1]");
    if (batch <= 0) return QB_OK;
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    Ham* ham = find_ham(ctx, ham_id);
    if (!ham) return fail(QB_ERR_NOT_FOUND, "unknown Hamiltonian id");
    if (!ham->diagonal) return fail(QB_ERR_INVALID, "CVaR needs a diagonal Hamiltonian; this one has non-diagonal terms");
    // every chunk below is launched against order data of 2^first->n_eff entries: all plans must match it and the Hamiltonian
    const Plan* first = nullptr;
    QB_TRY(check_plans(ctx, batch, plan_ids, ham->n_qubits, "Hamiltonian acts", "CVaR", &first));
    // alpha ~ 1 (numpy.isclose(alpha, 1)): the greedy fill in basis order, no sort (expectation.lower_tail_expectation_arrays)
    const bool sorted = std::fabs(alpha - 1.0) > 1e-8 + 1e-5;
    QB_TRY(ensure_cvar_order(ctx, *ham, first->n_eff, sorted));
    const uint32_t* perm = sorted ? ham->cvar_perm.as<uint32_t>() : nullptr;
    const double* energy = sorted ? ham->cvar_sorted.as<double>() : ham->cvar_energy.as<double>();
    // the statevectors share the workspace with the CVaR data the Hamiltonian holds
    const size_t state_bytes = (size_t(1) << first->n_eff) * amp_bytes(first->dtype);
    const size_t limit = workspace_limit_of(ctx), kept = ham->cvar_energy.cap + ham->cvar_perm.cap + ham->cvar_sorted.cap;
    if (kept + state_bytes > limit)
        return fail(QB_ERR_MEMORY, "CVaR data (" + std::to_string(kept) + " bytes) and one statevector (" + std::to_string(state_bytes) +
                                       " bytes) do not fit the workspace of " + std::to_string(limit) + " bytes");
    const int chunk = int(std::min<size_t>({size_t(batch), max_batch_for(ctx, first), (limit - kept) / state_bytes}));
    return run_oneshot(ctx, batch, plan_ids, params, param_offsets, nullptr, chunk, [&](DeviceBatch& b, int lo) {
        const int n = b.batch;
        const uint64_t size = uint64_t(1) << b.n_eff;
        const uint64_t n_chunks = size >> qb::kChunkBits;
        QB_TRY(ctx->scratch.reserve(sizeof(double) * (2 * size_t(n) * n_chunks + size_t(n))));
        double* d_mass = ctx->scratch.as<double>();
        double* d_pe = d_mass + size_t(n) * n_chunks;  // right after the masses: one scan launch covers both
        double* d_out = d_pe + size_t(n) * n_chunks;
        dim3 cgrid(unsigned(std::min<uint64_t>((n_chunks + 7) / 8, 2048)), unsigned(n));
        const unsigned fgrid = unsigned((n + 7) / 8);
        QB_TRY(with_dtype(b.dtype, [&](auto t) {
            using T = decltype(t);
            using C = typename qb::Cx<T>::type;
            qb::cvar_chunk_kernel<T><<<cgrid, 256, 0, ctx->stream>>>(b.states.as<C>(), size, perm, energy, n_chunks, d_mass, d_pe);
            QB_TRY(check_launch(ctx, "cvar_chunk_kernel"));
            qb::scan_chunks_kernel<<<2 * n, 1024, 0, ctx->stream>>>(d_mass, n_chunks);
            QB_TRY(check_launch(ctx, "scan_chunks_kernel"));
            qb::cvar_finish_kernel<T><<<fgrid, 256, 0, ctx->stream>>>(b.states.as<C>(), size, perm, energy, d_mass, d_pe, n_chunks, alpha, n, d_out);
            return check_launch(ctx, "cvar_finish_kernel");
        }));
        QB_TRY(ctx->pin_out.reserve(sizeof(double) * size_t(n)));
        QB_CUDA(cudaMemcpyAsync(ctx->pin_out.p, d_out, sizeof(double) * size_t(n), cudaMemcpyDeviceToHost, ctx->stream));
        QB_CUDA(cudaStreamSynchronize(ctx->stream));
        scatter_rows(out_values + lo, ctx->pin_out.p, b.order, sizeof(double));
        return QB_OK;
    });
}

int qb_evaluate_observables(qb_context* ctx, int batch, const int64_t* plan_ids, const double* params, const int64_t* param_offsets,
                            int64_t obs_id, double* out_values) {
    if (!ctx || !plan_ids || !param_offsets || !out_values) return fail(QB_ERR_INVALID, "null argument");
    if (batch <= 0) return QB_OK;
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    const Obs* ob = find_obs(ctx, obs_id);
    if (!ob) return fail(QB_ERR_NOT_FOUND, "unknown observable set id");
    const Plan* first = nullptr;
    QB_TRY(check_plans(ctx, batch, plan_ids, ob->n_qubits, "observables act", "observables", &first));
    // per state: the statevector, its string values, its observable values and the partials of at least one string
    const uint64_t size = uint64_t(1) << first->n_eff;
    const uint64_t count = std::max<uint64_t>(size >> qb::kExpTileBits, std::min<uint64_t>(1024, std::max<uint64_t>(1, size / 256)));
    const size_t state_bytes = size_t(size) * amp_bytes(first->dtype);
    const size_t values_bytes = sizeof(double) * (size_t(ob->n_terms) + size_t(ob->n_obs));
    const size_t per_state = state_bytes + values_bytes + sizeof(double) * size_t(count);
    const size_t limit = workspace_limit_of(ctx);
    if (per_state > limit)
        return fail(QB_ERR_MEMORY, "one statevector (" + std::to_string(state_bytes) + " bytes) and its observable scratch (" +
                                       std::to_string(per_state - state_bytes) + " bytes) do not fit the workspace of " + std::to_string(limit) + " bytes");
    const int chunk = int(std::min<size_t>({size_t(batch), max_batch_for(ctx, first), limit / per_state}));
    const size_t n_out = size_t(ob->n_obs);
    return run_oneshot(ctx, batch, plan_ids, params, param_offsets, nullptr, chunk, [&](DeviceBatch& b, int lo) {
        const int n = b.batch;
        const size_t terms_bytes = sizeof(double) * size_t(n) * size_t(ob->n_terms), out_bytes = sizeof(double) * size_t(n) * n_out;
        const size_t room = limit - size_t(n) * state_bytes - terms_bytes - out_bytes;  // >= n * count * 8 by the chunk size
        const size_t partial_bytes = std::max(sizeof(double) * size_t(count) * size_t(n), std::min(kTermPartialBytes, room));
        QB_TRY(ctx->scratch.reserve(terms_bytes + out_bytes + partial_bytes + 16));
        double* d_terms = ctx->scratch.as<double>();
        double* d_out = d_terms + size_t(n) * size_t(ob->n_terms);
        double* d_partials = d_out + size_t(n) * n_out;
        QB_TRY(with_dtype(b.dtype, [&](auto t) { return launch_terms_t<decltype(t)>(ctx, b, *ob, d_partials, partial_bytes, d_terms); }));
        qb::combine_observables_kernel<<<dim3(unsigned((n_out + 127) / 128), unsigned(n)), 128, 0, ctx->stream>>>(
            d_terms, ob->n_terms, ob->row_begin.as<int64_t>(), ob->cols.as<int32_t>(), ob->coeff.as<double>(), ob->n_obs, d_out);
        QB_TRY(check_launch(ctx, "combine_observables_kernel"));
        QB_TRY(ctx->pin_out.reserve(out_bytes));
        QB_CUDA(cudaMemcpyAsync(ctx->pin_out.p, d_out, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        QB_CUDA(cudaStreamSynchronize(ctx->stream));
        scatter_rows(out_values + size_t(lo) * n_out, ctx->pin_out.p, b.order, sizeof(double) * n_out);
        return QB_OK;
    });
}

// ---- most probable basis states ------------------------------------------------------------------------
int qb_top_select_init(qb_top_select* sel, int n_qubits, int64_t max_states) {
    if (!sel) return fail(QB_ERR_INVALID, "null select state");
    if (n_qubits < 1 || n_qubits > 63) return fail(QB_ERR_INVALID, "n_qubits must be in 1..63");
    QB_TRY(check_top_limits(max_states, 0.0));
    *sel = qb_top_select{};
    sel->max_states = sel->need = uint64_t(max_states);
    sel->n_qubits = n_qubits, sel->p_free = 64, sel->idx_hi = n_qubits;
    return QB_OK;
}

// The decision rule of every route.  The buckets of this pass partition the entries of the current prefix range, in key order;
// the first bucket at which the running count reaches `need` holds the cut.  Reached exactly: the bucket is taken whole and
// the stop key is its last key.  Otherwise the bucket's digit is fixed and the next pass splits it.
int qb_top_select_pick(qb_top_select* sel, const uint64_t counts[256]) {
    if (!counts) return fail(QB_ERR_INVALID, "null counts");
    QB_TRY(check_top_state(sel, nullptr, false));
    qb_top_select& s = *sel;
    uint64_t total = 0;
    for (int b = 0; b < qb::kSelBuckets; ++b) total += counts[b];
    const bool first = s.passes == 0;
    s.passes++;
    if (total <= s.need) {
        if (!first) return fail(QB_ERR_INVALID, "the bucket counts of a later pass must exceed the entries still needed");
        s.done = 1, s.selected = total;  // no more eligible entries than max_states: all of them
        s.stop_key = s.stop_index = ~uint64_t(0);
        return QB_OK;
    }
    int pick = 0;
    uint64_t before = 0;
    while (before + counts[pick] < s.need) before += counts[pick++];
    const bool whole = before + counts[pick] == s.need;
    if (s.p_free > 0) {
        const int low = s.p_free - qb::kSelBits;
        const uint64_t fixed = (s.p_free == 64 ? 0 : s.p_prefix << s.p_free) | (uint64_t(pick) << low);
        if (whole) {
            s.stop_key = fixed | ((uint64_t(1) << low) - 1), s.stop_index = ~uint64_t(0);
        } else {
            s.p_prefix = (s.p_free == 64 ? 0 : s.p_prefix << qb::kSelBits) | uint64_t(pick);
            s.p_free = low;
        }
    } else {
        const int lo = std::max(0, s.idx_hi - qb::kSelBits);
        if (pick >> (s.idx_hi - lo)) return fail(QB_ERR_INVALID, "a count in a bucket beyond the digit's width");
        const uint64_t fixed = s.idx_prefix | (uint64_t(pick) << lo);
        if (whole) {
            s.stop_key = s.p_prefix, s.stop_index = fixed | ((uint64_t(1) << lo) - 1);
        } else {
            if (lo == 0) return fail(QB_ERR_INVALID, "more than one entry counted for one complete key");
            s.idx_prefix = fixed, s.idx_hi = lo;
        }
    }
    if (whole) {
        s.done = 1, s.selected = s.max_states;
    } else {
        s.taken += before, s.need -= before;
    }
    return QB_OK;
}

int qb_top_states(qb_context* ctx, int batch, const int64_t* plan_ids, const double* params, const int64_t* param_offsets, int64_t max_states,
                  double min_probability, int64_t* out_counts, int64_t* out_indices, double* out_probs) {
    if (!ctx || !plan_ids || !param_offsets || !out_counts || !out_indices || !out_probs) return fail(QB_ERR_INVALID, "null argument");
    QB_TRY(check_top_limits(max_states, min_probability));
    if (batch <= 0) return QB_OK;
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    const Plan* first = find_plan(ctx, plan_ids[0]);
    if (!first) return fail(QB_ERR_NOT_FOUND, "unknown plan id " + std::to_string(plan_ids[0]));
    QB_TRY(check_plans(ctx, batch, plan_ids, first->n_qubits, "the first circuit acts", "top-states", &first));
    const uint64_t size = uint64_t(1) << first->n_eff, M = uint64_t(max_states);
    uint64_t seg = 0;
    const unsigned col_ctas = top_collect_ctas(ctx, size, &seg);
    // per state: the statevector, its output rows (16 B per slot), its bucket counts, per-CTA counts and pass arguments; once:
    // the sort's second buffers and CUB's storage
    size_t sort_bytes = 0;
    {
        cub::DoubleBuffer<double> keys(nullptr, nullptr);
        cub::DoubleBuffer<int64_t> vals(nullptr, nullptr);
        QB_CUDA(cub::DeviceRadixSort::SortPairsDescending(nullptr, sort_bytes, keys, vals, int(M), 0, 64, ctx->stream));
    }
    auto align = [](size_t v) { return (v + 255) & ~size_t(255); };
    const size_t state_bytes = size_t(size) * amp_bytes(first->dtype);
    const size_t row_bytes = align(16 * M) + align(sizeof(uint64_t) * qb::kSelBuckets) + align(sizeof(uint32_t) * col_ctas) +
                             align(sizeof(qb::TopSelectArgs)) + align(sizeof(qb::TopCollectArgs));
    const size_t once_bytes = align(16 * M) + align(sort_bytes);
    const size_t limit = workspace_limit_of(ctx);
    if (state_bytes + row_bytes + once_bytes > limit)
        return fail(QB_ERR_MEMORY, "one statevector (" + std::to_string(state_bytes) + " bytes) and its top-states scratch (" +
                                       std::to_string(row_bytes + once_bytes) + " bytes) do not fit the workspace of " + std::to_string(limit) + " bytes");
    const int chunk = int(std::min<size_t>({size_t(batch), max_batch_for(ctx, first), (limit - once_bytes) / (state_bytes + row_bytes)}));
    return run_oneshot(ctx, batch, plan_ids, params, param_offsets, nullptr, chunk, [&](DeviceBatch& b, int lo) {
        const int n = b.batch;
        const size_t nn = size_t(n);
        size_t at = 0;
        auto carve = [&](size_t bytes) {
            const size_t here = at;
            at += align(bytes);
            return here;
        };
        const size_t o_counts = carve(sizeof(uint64_t) * qb::kSelBuckets * nn), o_cta = carve(sizeof(uint32_t) * col_ctas * nn);
        const size_t o_idx = carve(sizeof(int64_t) * M * nn), o_prob = carve(sizeof(double) * M * nn);
        const size_t o_alt_idx = carve(sizeof(int64_t) * M), o_alt_prob = carve(sizeof(double) * M);
        const size_t o_sel = carve(sizeof(qb::TopSelectArgs) * nn), o_col = carve(sizeof(qb::TopCollectArgs) * nn), o_temp = carve(sort_bytes);
        QB_TRY(ctx->scratch.reserve(at));
        unsigned char* base = static_cast<unsigned char*>(ctx->scratch.p);
        auto* d_counts = reinterpret_cast<unsigned long long*>(base + o_counts);
        auto* d_cta = reinterpret_cast<uint32_t*>(base + o_cta);
        auto* d_idx = reinterpret_cast<int64_t*>(base + o_idx);
        auto* d_prob = reinterpret_cast<double*>(base + o_prob);
        auto* d_sel = reinterpret_cast<qb::TopSelectArgs*>(base + o_sel);
        auto* d_col = reinterpret_cast<qb::TopCollectArgs*>(base + o_col);
        std::vector<qb_top_select> sel(nn);
        for (auto& s : sel) QB_TRY(qb_top_select_init(&s, b.n_qubits, max_states));
        // the select: every unfinished state of the chunk in each pass, one synchronisation per pass
        std::vector<qb::TopSelectArgs> args;
        std::vector<int> rows;
        std::vector<uint64_t> counts;
        for (;;) {
            args.clear(), rows.clear();
            for (int i = 0; i < n; ++i)
                if (!sel[i].done) args.push_back(top_select_args(sel[i], nullptr, min_probability, i)), rows.push_back(i);
            if (rows.empty()) break;
            const int m = int(rows.size());
            counts.resize(size_t(m) * qb::kSelBuckets);
            QB_TRY(with_dtype(b.dtype, [&](auto t) {
                return top_select_pass_t<decltype(t)>(ctx, b.states.p, size, size, b.n_eff, 0, args.data(), m, d_sel, d_counts, counts.data());
            }));
            for (int r = 0; r < m; ++r) QB_TRY(qb_top_select_pick(&sel[rows[r]], counts.data() + size_t(r) * qb::kSelBuckets));
        }
        std::vector<qb::TopCollectArgs> cargs(nn);
        for (int i = 0; i < n; ++i) cargs[i] = top_collect_args(sel[i], nullptr, min_probability, i);
        std::vector<uint64_t> totals;
        QB_TRY(with_dtype(b.dtype, [&](auto t) {
            return top_collect_t<decltype(t)>(ctx, b.states.p, size, size, b.n_eff, 0, cargs.data(), n, d_col, d_cta, M, d_idx, d_prob, totals);
        }));
        // per state: stable sort by descending p (the collect wrote index order), then its row straight into the caller's arrays
        for (int pos = 0; pos < n; ++pos) {
            if (totals[pos] != sel[pos].selected)
                return fail(QB_ERR_CUDA, "the collect found " + std::to_string(totals[pos]) + " entries, the select " + std::to_string(sel[pos].selected));
            const int cnt = int(totals[pos]);
            cub::DoubleBuffer<double> keys(d_prob + size_t(pos) * M, reinterpret_cast<double*>(base + o_alt_prob));
            cub::DoubleBuffer<int64_t> vals(d_idx + size_t(pos) * M, reinterpret_cast<int64_t*>(base + o_alt_idx));
            if (cnt > 1) QB_CUDA(cub::DeviceRadixSort::SortPairsDescending(base + o_temp, sort_bytes, keys, vals, cnt, 0, 64, ctx->stream));
            const size_t row = size_t(lo) + size_t(b.order[pos]);
            int64_t* idx_row = out_indices + row * M;
            double* prob_row = out_probs + row * M;
            if (cnt) {
                QB_CUDA(cudaMemcpyAsync(idx_row, vals.Current(), sizeof(int64_t) * cnt, cudaMemcpyDeviceToHost, ctx->stream));
                QB_CUDA(cudaMemcpyAsync(prob_row, keys.Current(), sizeof(double) * cnt, cudaMemcpyDeviceToHost, ctx->stream));
            }
            QB_CUDA(cudaStreamSynchronize(ctx->stream));  // (the second buffers serve the next state)
            std::fill(idx_row + cnt, idx_row + M, int64_t(-1));
            std::fill(prob_row + cnt, prob_row + M, 0.0);
            out_counts[row] = cnt;
        }
        return QB_OK;
    });
}

// ---- exact marginal probabilities ------------------------------------------------------------------------
int qb_marginal_probabilities(qb_context* ctx, int batch, const int64_t* plan_ids, const double* params, const int64_t* param_offsets, int n_measured,
                              const int* qubits, double* out) {
    if (!ctx || !plan_ids || !param_offsets || !qubits || !out) return fail(QB_ERR_INVALID, "null argument");
    if (n_measured < 1 || n_measured > qb::kMargMaxBits)
        return fail(QB_ERR_INVALID, "n_measured must be in 1.." + std::to_string(qb::kMargMaxBits) + ", got " + std::to_string(n_measured));
    if (batch <= 0) return QB_OK;
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    const Plan* first = find_plan(ctx, plan_ids[0]);
    if (!first) return fail(QB_ERR_NOT_FOUND, "unknown plan id " + std::to_string(plan_ids[0]));
    QB_TRY(check_plans(ctx, batch, plan_ids, first->n_qubits, "the first circuit acts", "marginal", &first));
    qb::MarginalArgs a;
    QB_TRY(marginal_args(first->n_eff, 0, n_measured, qubits, first->n_qubits, &a));
    const uint64_t size = uint64_t(1) << first->n_eff;
    const size_t state_bytes = size_t(size) * amp_bytes(first->dtype), row_bytes = marginal_scratch_bytes(a);
    const size_t limit = workspace_limit_of(ctx);
    if (state_bytes + row_bytes > limit)
        return fail(QB_ERR_MEMORY, "one statevector (" + std::to_string(state_bytes) + " bytes) and its marginal scratch (" + std::to_string(row_bytes) +
                                       " bytes) do not fit the workspace of " + std::to_string(limit) + " bytes");
    const int chunk = int(std::min<size_t>({size_t(batch), max_batch_for(ctx, first), limit / (state_bytes + row_bytes)}));
    const size_t out_row = size_t(1) << n_measured;
    return run_oneshot(ctx, batch, plan_ids, params, param_offsets, nullptr, chunk, [&](DeviceBatch& b, int lo) {
        const size_t nn = size_t(b.batch);
        QB_TRY(ctx->scratch.reserve(nn * row_bytes));
        double* d_out = ctx->scratch.as<double>();
        double* d_part = d_out + nn * out_row;
        QB_TRY(with_dtype(b.dtype, [&](auto t) { return marginal_t<decltype(t)>(ctx, b.states.p, size, b.batch, b.n_eff, a, d_part, d_out); }));
        for (size_t pos = 0; pos < nn; ++pos)
            QB_CUDA(cudaMemcpyAsync(out + (size_t(lo) + size_t(b.order[pos])) * out_row, d_out + pos * out_row, sizeof(double) * out_row,
                                    cudaMemcpyDeviceToHost, ctx->stream));
        QB_CUDA(cudaStreamSynchronize(ctx->stream));
        return QB_OK;
    });
}

int qb_marginal_device(qb_context* ctx, int dtype, int n_local, const void* d_state, uint64_t index_offset, int n_measured, const int* qubits,
                       double* out) {
    if (!ctx || !d_state || !qubits || !out) return fail(QB_ERR_INVALID, "null argument");
    if (n_local < 8 || n_local > 36) return fail(QB_ERR_INVALID, "n_local out of range");
    if (dtype != QB_C128 && dtype != QB_C64) return fail(QB_ERR_INVALID, "dtype must be QB_C128 or QB_C64");
    if (index_offset & ((uint64_t(1) << n_local) - 1)) return fail(QB_ERR_INVALID, "index_offset has bits below n_local");
    qb::MarginalArgs a;
    QB_TRY(marginal_args(n_local, index_offset, n_measured, qubits, 64, &a));
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    QB_TRY(ctx->scratch.reserve(marginal_scratch_bytes(a)));
    double* d_out = ctx->scratch.as<double>();
    double* d_part = d_out + (size_t(1) << n_measured);
    const uint64_t size = uint64_t(1) << n_local;
    QB_TRY(with_dtype(dtype, [&](auto t) { return marginal_t<decltype(t)>(ctx, d_state, size, 1, n_local, a, d_part, d_out); }));
    QB_CUDA(cudaMemcpyAsync(out, d_out, sizeof(double) << n_measured, cudaMemcpyDeviceToHost, ctx->stream));
    QB_CUDA(cudaStreamSynchronize(ctx->stream));
    return QB_OK;
}

int qb_statevector(qb_context* ctx, int64_t plan_id, const double* params, int n_params, double* out_re_im) {
    if (!ctx || !out_re_im) return fail(QB_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    Plan* pl = find_plan(ctx, plan_id);
    if (!pl) return fail(QB_ERR_NOT_FOUND, "unknown plan id");
    DeviceBatch& b = ctx->oneshot;
    QB_TRY(build_batch(ctx, b, 1, &plan_id, nullptr, nullptr, 1, 0));
    const int64_t offs[2] = {0, n_params};
    QB_TRY(batch_upload_params(ctx, b, params, offs));
    QB_TRY(launch_circuits(ctx, b, nullptr));
    const uint64_t size = uint64_t(1) << pl->n_qubits;
    const void* src = b.states.p;
    if (pl->dtype == QB_C64) {
        QB_TRY(ctx->scratch.reserve(sizeof(double2) * size));
        qb::to_c128_kernel<float><<<int(std::min<uint64_t>(1024, (size + 255) / 256)), 256, 0, ctx->stream>>>(b.states.as<float2>(),
                                                                                                              ctx->scratch.as<double2>(), size);
        QB_TRY(check_launch(ctx, "to_c128_kernel"));
        src = ctx->scratch.p;
    }
    QB_CUDA(cudaMemcpyAsync(out_re_im, src, sizeof(double2) * size, cudaMemcpyDeviceToHost, ctx->stream));
    QB_CUDA(cudaStreamSynchronize(ctx->stream));
    return QB_OK;
}

// ---- device-pointer entry points -----------------------------------------------------------------------
int qb_apply_plan_device(qb_context* ctx, int64_t plan_id, const double* params_host, int n_params, void* d_state, int init_zero_state,
                         uint64_t index_offset) {
    if (!ctx || !d_state) return fail(QB_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    const Plan* pl = find_plan(ctx, plan_id);
    if (!pl) return fail(QB_ERR_NOT_FOUND, "unknown plan id");
    // the sweeps cover 2^n_eff amplitudes; a caller-owned state holds exactly 2^n_qubits
    if (pl->n_eff != pl->n_qubits)
        return fail(QB_ERR_INVALID, "a caller-owned state of " + std::to_string(pl->n_qubits) + " qubits is smaller than one " +
                                        std::to_string(pl->n_eff) + "-qubit sweep tile");
    DeviceBatch b;
    QB_TRY(build_batch(ctx, b, 1, &plan_id, nullptr, d_state, init_zero_state, index_offset));
    const int64_t offs[2] = {0, n_params};
    QB_TRY(batch_upload_params(ctx, b, params_host, offs));
    QB_TRY(launch_circuits(ctx, b, nullptr));
    QB_CUDA(cudaStreamSynchronize(ctx->stream));
    return QB_OK;
}

int qb_expectation_device(qb_context* ctx, int64_t ham_id, int dtype, int n_local, const void* d_state, uint64_t index_offset,
                          double* out_value) {
    if (!ctx || !d_state || !out_value) return fail(QB_ERR_INVALID, "null argument");
    if (n_local < 8 || n_local > 36) return fail(QB_ERR_INVALID, "n_local out of range");
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    Ham* ham = find_ham(ctx, ham_id);
    if (!ham) return fail(QB_ERR_NOT_FOUND, "unknown Hamiltonian id");
    const size_t n_part = std::max<size_t>(1024, n_local >= qb::kExpTileBits ? size_t(1) << (n_local - qb::kExpTileBits) : 0);
    QB_TRY(ctx->scratch.reserve(sizeof(double) * (n_part + 16)));
    double* d_part = ctx->scratch.as<double>();
    double* d_out = d_part + n_part;
    QB_TRY(with_dtype(dtype, [&](auto t) { return expectation_state_t<decltype(t)>(ctx, *ham, d_state, n_local, index_offset, d_part, d_out); }));
    QB_CUDA(cudaMemcpyAsync(out_value, d_out, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    QB_CUDA(cudaStreamSynchronize(ctx->stream));
    return QB_OK;
}

int qb_sample_device(qb_context* ctx, int dtype, int n_local, const void* d_state, int shots, const double* uniforms, int64_t* out_indices) {
    if (!ctx || !d_state || !uniforms || !out_indices) return fail(QB_ERR_INVALID, "null argument");
    if (shots <= 0) return QB_OK;
    if (n_local < qb::kChunkBits || n_local > 36) return fail(QB_ERR_INVALID, "n_local out of range");
    if (dtype != QB_C128 && dtype != QB_C64) return fail(QB_ERR_INVALID, "dtype must be QB_C128 or QB_C64");
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    const uint64_t size = uint64_t(1) << n_local;
    const uint64_t n_chunks = size >> qb::kChunkBits;
    const size_t u_bytes = sizeof(double) * size_t(shots);
    QB_TRY(ctx->scratch.reserve(2 * u_bytes + sizeof(double) * n_chunks));
    double* d_uniforms = ctx->scratch.as<double>();
    int64_t* d_indices = reinterpret_cast<int64_t*>(d_uniforms + shots);
    double* d_chunks = reinterpret_cast<double*>(d_indices + shots);
    QB_CUDA(cudaMemcpyAsync(d_uniforms, uniforms, u_bytes, cudaMemcpyHostToDevice, ctx->stream));
    QB_TRY(with_dtype(dtype, [&](auto t) {
        using T = decltype(t);
        return launch_sampling_t<T>(ctx, static_cast<const typename qb::Cx<T>::type*>(d_state), size, 1, size, d_uniforms, shots, d_chunks, d_indices);
    }));
    QB_CUDA(cudaMemcpyAsync(out_indices, d_indices, u_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    QB_CUDA(cudaStreamSynchronize(ctx->stream));
    return QB_OK;
}

int qb_cvar_select_device(qb_context* ctx, int64_t ham_id, int dtype, int n_local, const void* d_state, uint64_t index_offset, void* d_cache,
                          int cache_mode, uint64_t e_prefix, int e_free, int digit_kind, int digit_bits, const int32_t* digit_positions,
                          uint64_t idx_mask, uint64_t idx_value, double* out_sums, uint64_t* out_ints) {
    if (!ctx || !out_sums || !out_ints || (cache_mode != 2 && !d_state)) return fail(QB_ERR_INVALID, "null argument");
    if (n_local < 8 || n_local > 36) return fail(QB_ERR_INVALID, "n_local out of range");
    if (dtype != QB_C128 && dtype != QB_C64) return fail(QB_ERR_INVALID, "dtype must be QB_C128 or QB_C64");
    if (cache_mode < 0 || cache_mode > 2 || (cache_mode && !d_cache)) return fail(QB_ERR_INVALID, "cache_mode must be 0, or 1 / 2 with a cache buffer");
    if (digit_bits < 1 || digit_bits > qb::kSelBits) return fail(QB_ERR_INVALID, "digit_bits must be in 1.." + std::to_string(qb::kSelBits));
    if (e_free < 0 || e_free > 64) return fail(QB_ERR_INVALID, "e_free must be in 0..64");
    if (e_free > 0 && e_free < 64 && (e_prefix >> (64 - e_free)) != 0) return fail(QB_ERR_INVALID, "e_prefix has bits beyond 64 - e_free");
    if ((idx_value & ~idx_mask) != 0) return fail(QB_ERR_INVALID, "idx_value has bits outside idx_mask");
    qb::SelectArgs a{};
    a.e_prefix = e_prefix, a.idx_mask = idx_mask, a.idx_value = idx_value, a.e_free = e_free, a.digit_kind = digit_kind, a.bits = digit_bits;
    if (digit_kind == 0) {
        if (e_free < digit_bits) return fail(QB_ERR_INVALID, "energy digit below the energy key's open bits");
    } else if (digit_kind == 1) {
        if (!digit_positions) return fail(QB_ERR_INVALID, "null digit_positions");
        uint64_t seen = idx_mask;
        for (int j = 0; j < digit_bits; ++j) {
            const int p = digit_positions[j];
            if (p < 0 || p > 63 || ((seen >> p) & 1)) return fail(QB_ERR_INVALID, "bad bit map: digit positions must be distinct, unfixed bit positions");
            seen |= uint64_t(1) << p;
            a.pos[j] = p;
        }
    } else {
        return fail(QB_ERR_INVALID, "digit_kind must be 0 (energy) or 1 (logical index)");
    }
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    Ham* ham = find_ham(ctx, ham_id);
    if (!ham) return fail(QB_ERR_NOT_FOUND, "unknown Hamiltonian id");
    if (!ham->diagonal) return fail(QB_ERR_INVALID, "CVaR needs a diagonal Hamiltonian; this one has non-diagonal terms");
    const uint64_t size = uint64_t(1) << n_local;
    // the grid depends on the device and the shard size only: the CTA-order reduction is the same on every call
    const int n_cta = int(std::min<uint64_t>(uint64_t(ctx->sm_count) * 4, std::max<uint64_t>(1, size / (32 * qb::kSelWarps * 16))));
    constexpr int B = qb::kSelBuckets;
    const size_t part_bytes = sizeof(double) * 2 * B * size_t(n_cta), sums_bytes = sizeof(double) * 2 * B, ints_bytes = sizeof(uint64_t) * 4 * B;
    QB_TRY(ctx->scratch.reserve(part_bytes + sums_bytes + ints_bytes));
    double* d_part = ctx->scratch.as<double>();
    double* d_sums = d_part + 2 * B * size_t(n_cta);
    unsigned long long* d_ints = reinterpret_cast<unsigned long long*>(d_sums + 2 * B);
    QB_CUDA(cudaMemsetAsync(d_ints, 0, sizeof(uint64_t) * B, ctx->stream));                  // count
    QB_CUDA(cudaMemsetAsync(d_ints + B, 0xff, sizeof(uint64_t) * B, ctx->stream));           // emin
    QB_CUDA(cudaMemsetAsync(d_ints + 2 * B, 0, sizeof(uint64_t) * B, ctx->stream));          // emax
    QB_CUDA(cudaMemsetAsync(d_ints + 3 * B, 0xff, sizeof(uint64_t) * B, ctx->stream));       // kmin
    const uint64_t* z = ham->diag_z.as<uint64_t>();
    const double* c = ham->diag_c.as<double>();
    double2* cache = static_cast<double2*>(d_cache);
    QB_TRY(with_dtype(dtype, [&](auto t) {
        using T = decltype(t);
        qb::cvar_select_kernel<T><<<n_cta, 32 * qb::kSelWarps, 0, ctx->stream>>>(static_cast<const typename qb::Cx<T>::type*>(d_state), cache, cache_mode,
                                                                                  size, index_offset, z, c, ham->n_diag, a, d_part, d_part + B * size_t(n_cta), d_ints);
        return check_launch(ctx, "cvar_select_kernel");
    }));
    qb::cvar_select_reduce_kernel<<<2 * B, 256, 0, ctx->stream>>>(d_part, n_cta, d_sums);
    QB_TRY(check_launch(ctx, "cvar_select_reduce_kernel"));
    QB_TRY(ctx->pin_out.reserve(sums_bytes + ints_bytes));
    QB_CUDA(cudaMemcpyAsync(ctx->pin_out.p, d_sums, sums_bytes + ints_bytes, cudaMemcpyDeviceToHost, ctx->stream));  // d_ints follows d_sums
    QB_CUDA(cudaStreamSynchronize(ctx->stream));
    std::memcpy(out_sums, ctx->pin_out.p, sums_bytes);
    std::memcpy(out_ints, static_cast<const unsigned char*>(ctx->pin_out.p) + sums_bytes, ints_bytes);
    return QB_OK;
}

int qb_top_select_device(qb_context* ctx, int dtype, int n_local, const void* d_state, uint64_t index_offset, double min_probability,
                         const qb_top_select* sel, const int32_t* positions, uint64_t* out_counts) {
    if (!out_counts) return fail(QB_ERR_INVALID, "null argument");
    QB_TRY(check_top_shard(ctx, dtype, n_local, d_state, min_probability, sel, positions, false));
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    const qb::TopSelectArgs args = top_select_args(*sel, positions, min_probability, 0);
    QB_TRY(ctx->scratch.reserve(sizeof(uint64_t) * qb::kSelBuckets + sizeof(qb::TopSelectArgs)));
    auto* d_counts = ctx->scratch.as<unsigned long long>();
    auto* d_args = reinterpret_cast<qb::TopSelectArgs*>(d_counts + qb::kSelBuckets);
    const uint64_t size = uint64_t(1) << n_local;
    return with_dtype(dtype, [&](auto t) {
        return top_select_pass_t<decltype(t)>(ctx, d_state, size, size, n_local, index_offset, &args, 1, d_args, d_counts, out_counts);
    });
}

int qb_top_collect_device(qb_context* ctx, int dtype, int n_local, const void* d_state, uint64_t index_offset, double min_probability,
                          const qb_top_select* sel, const int32_t* positions, int64_t capacity, int64_t* out_count, int64_t* out_indices,
                          double* out_probs) {
    if (!out_count || !out_indices || !out_probs) return fail(QB_ERR_INVALID, "null argument");
    if (capacity < 0) return fail(QB_ERR_INVALID, "negative capacity");
    QB_TRY(check_top_shard(ctx, dtype, n_local, d_state, min_probability, sel, positions, true));
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    const qb::TopCollectArgs args = top_collect_args(*sel, positions, min_probability, 0);
    const uint64_t size = uint64_t(1) << n_local, cap = uint64_t(std::max<int64_t>(capacity, 1));
    uint64_t seg = 0;
    const unsigned n_cta = top_collect_ctas(ctx, size, &seg);
    const size_t idx_bytes = sizeof(int64_t) * cap, cta_bytes = (sizeof(uint32_t) * n_cta + 15) & ~size_t(15);
    QB_TRY(ctx->scratch.reserve(2 * idx_bytes + cta_bytes + sizeof(qb::TopCollectArgs)));
    auto* d_idx = ctx->scratch.as<int64_t>();
    auto* d_prob = reinterpret_cast<double*>(d_idx + cap);
    auto* d_cta = reinterpret_cast<uint32_t*>(d_prob + cap);
    auto* d_args = reinterpret_cast<qb::TopCollectArgs*>(reinterpret_cast<unsigned char*>(d_cta) + cta_bytes);
    std::vector<uint64_t> totals;
    QB_TRY(with_dtype(dtype, [&](auto t) {
        return top_collect_t<decltype(t)>(ctx, d_state, size, size, n_local, index_offset, &args, 1, d_args, d_cta, uint64_t(capacity), d_idx, d_prob, totals);
    }));
    if (totals[0]) {
        QB_CUDA(cudaMemcpyAsync(out_indices, d_idx, sizeof(int64_t) * totals[0], cudaMemcpyDeviceToHost, ctx->stream));
        QB_CUDA(cudaMemcpyAsync(out_probs, d_prob, sizeof(double) * totals[0], cudaMemcpyDeviceToHost, ctx->stream));
    }
    QB_CUDA(cudaStreamSynchronize(ctx->stream));
    *out_count = int64_t(totals[0]);
    return QB_OK;
}

int qb_swap_global_p2p(qb_context* ctx, int dtype, int n_local, const void* d_state, void* const* peer_dst, int world, int rank, int n_global,
                       const int32_t* local_positions) {
    if (!ctx || !d_state || !peer_dst || !local_positions) return fail(QB_ERR_INVALID, "null argument");
    if (dtype != QB_C128 && dtype != QB_C64) return fail(QB_ERR_INVALID, "dtype must be QB_C128 or QB_C64");
    if (n_global < 1 || n_global > 4 || world != (1 << n_global) || rank < 0 || rank >= world) return fail(QB_ERR_INVALID, "bad rank layout");
    if (n_local < n_global || n_local > 36) return fail(QB_ERR_INVALID, "n_local out of range");
    qb::SwapArgs args{};
    uint64_t seen = 0;
    for (int j = 0; j < n_global; ++j) {
        const int p = local_positions[j];
        if (p < 0 || p >= n_local || ((seen >> p) & 1) || (j && p <= local_positions[j - 1])) return fail(QB_ERR_INVALID, "local positions must be distinct, ascending and below n_local");
        seen |= 1ull << p;
        args.lp[j] = p;
    }
    for (int r = 0; r < world; ++r) {
        if (!peer_dst[r]) return fail(QB_ERR_INVALID, "null peer buffer");
        args.peer[r] = peer_dst[r];
    }
    args.g = n_global, args.rank = rank;
    args.run_bits = std::min(qb::kSwapRunBits, n_local - n_global);
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    const uint64_t size = uint64_t(1) << n_local;
    const int blocks = int(std::min<uint64_t>(uint64_t(ctx->sm_count) * 8, std::max<uint64_t>(1, size / (256 * 4))));
    return with_dtype(dtype, [&](auto t) {
        using C = typename qb::Cx<decltype(t)>::type;
        qb::swap_p2p_kernel<C><<<blocks, 256, 0, ctx->stream>>>(static_cast<const C*>(d_state), args, size);
        return check_launch(ctx, "swap_p2p_kernel");
    });
}

int qb_swap_global_inplace_p2p(qb_context* ctx, int dtype, int n_local, void* const* shard_states, int world, int rank, int n_global,
                               const int32_t* local_positions) {
    if (!ctx || !shard_states || !local_positions) return fail(QB_ERR_INVALID, "null argument");
    if (dtype != QB_C128 && dtype != QB_C64) return fail(QB_ERR_INVALID, "dtype must be QB_C128 or QB_C64");
    if (n_global < 1 || n_global > 4 || world != (1 << n_global) || rank < 0 || rank >= world) return fail(QB_ERR_INVALID, "bad rank layout");
    if (n_local < n_global + 1 || n_local > 36) return fail(QB_ERR_INVALID, "n_local out of range (the in-place exchange needs n_local >= n_global + 1)");
    qb::SwapInplaceArgs args{};
    uint64_t seen = 0;
    for (int j = 0; j < n_global; ++j) {
        const int p = local_positions[j];
        if (p < 0 || p >= n_local || ((seen >> p) & 1) || (j && p <= local_positions[j - 1])) return fail(QB_ERR_INVALID, "local positions must be distinct, ascending and below n_local");
        seen |= 1ull << p;
        args.lpmask |= 1ull << p;
        args.rbits |= uint64_t((rank >> j) & 1) << p;
    }
    for (int r = 0; r < world; ++r) {
        if (!shard_states[r]) return fail(QB_ERR_INVALID, "null shard buffer");
        args.state[r] = shard_states[r];
    }
    // the owner bit: the highest local position not exchanged (exists because n_local > n_global).  Any such bit partitions the
    // pairs; a high one keeps neighbouring pair numbers on neighbouring amplitudes (bit 0 would halve every sector's use).
    int p0 = n_local - 1;
    while ((seen >> p0) & 1) --p0;
    int s = 0;  // merge p0 into the ascending lp
    for (; s < n_global && local_positions[s] < p0; ++s) args.ins_pos[s] = local_positions[s], args.ins_src[s] = s;
    args.ins_pos[s] = p0, args.ins_src[s] = n_global;
    for (int j = s; j < n_global; ++j) args.ins_pos[j + 1] = local_positions[j], args.ins_src[j + 1] = j;
    args.g = n_global, args.rank = rank;
    args.run_bits = std::min(qb::kSwapRunBits, n_local - n_global - 1);
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    const uint64_t items = uint64_t(world - 1) << (n_local - n_global - 1);
    const int blocks = int(std::min<uint64_t>(uint64_t(ctx->sm_count) * 8, std::max<uint64_t>(1, items / (256 * qb::kInplaceUnroll))));
    return with_dtype(dtype, [&](auto t) {
        using C = typename qb::Cx<decltype(t)>::type;
        qb::swap_inplace_p2p_kernel<C><<<blocks, 256, 0, ctx->stream>>>(args, items);
        return check_launch(ctx, "swap_inplace_p2p_kernel");
    });
}

int qb_evaluate_expectation_submit(qb_context* ctx, int batch, const int64_t* plan_ids, const double* params, const int64_t* param_offsets,
                                   int64_t ham_id) {
    if (!ctx || !plan_ids || !param_offsets) return fail(QB_ERR_INVALID, "null argument");
    if (batch <= 0) return QB_OK;
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    Ham* ham = find_ham(ctx, ham_id);
    if (!ham) return fail(QB_ERR_NOT_FOUND, "unknown Hamiltonian id");
    Plan* first = find_plan(ctx, plan_ids[0]);
    if (!first) return fail(QB_ERR_NOT_FOUND, "unknown plan id " + std::to_string(plan_ids[0]));
    if (size_t(batch) > max_batch_for(ctx, first)) return fail(QB_ERR_MEMORY, "chunk does not fit the statevector workspace");
    const size_t need = sizeof(double) * (ctx->pending_results + size_t(batch));
    if (need > ctx->pin_res.cap) {  // grow the pinned result buffer: drain what is in flight first, keep its contents
        QB_CUDA(cudaStreamSynchronize(ctx->stream));
        std::vector<double> keep(ctx->pending_results);
        if (ctx->pending_results) std::memcpy(keep.data(), ctx->pin_res.p, sizeof(double) * ctx->pending_results);
        QB_TRY(ctx->pin_res.reserve(std::max<size_t>(2 * need, size_t(1) << 16)));
        if (ctx->pending_results) std::memcpy(ctx->pin_res.p, keep.data(), sizeof(double) * ctx->pending_results);
    }
    DeviceBatch& b = ctx->oneshot;
    QB_TRY(build_batch(ctx, b, batch, plan_ids, ham, nullptr, 1, 0));
    QB_TRY(batch_upload_params(ctx, b, params, param_offsets));
    QB_TRY(launch_circuits(ctx, b, nullptr));
    QB_TRY(launch_expectation(ctx, b));
    double* dst = static_cast<double*>(ctx->pin_res.p) + ctx->pending_results;
    QB_CUDA(cudaMemcpyAsync(dst, b.out.p, sizeof(double) * size_t(batch), cudaMemcpyDeviceToHost, ctx->stream));
    ctx->pending.push_back({ctx->pending_results, b.order});
    ctx->pending_results += size_t(batch);
    return QB_OK;
}

int qb_evaluate_expectation_collect(qb_context* ctx, int total, double* out_values) {
    if (!ctx || (total > 0 && !out_values)) return fail(QB_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    const size_t have = ctx->pending_results;
    std::vector<qb_context::PendingChunk> chunks;
    chunks.swap(ctx->pending);
    ctx->pending_results = 0;
    if (e != cudaSuccess) return fail(QB_ERR_CUDA, std::string("cudaStreamSynchronize: ") + cudaGetErrorString(e));
    if (size_t(total) != have) return fail(QB_ERR_INVALID, "collect asked for " + std::to_string(total) + " results, " + std::to_string(have) + " are pending");
    const double* res = static_cast<const double*>(ctx->pin_res.p);
    for (const auto& ch : chunks) scatter_rows(out_values + ch.offset, res + ch.offset, ch.order, sizeof(double));
    return QB_OK;
}

int qb_evaluate_expectation_multi(int n_ctx, qb_context* const* ctxs, const int* batches, const int64_t* const* plan_ids,
                                  const double* const* params, const int64_t* const* param_offsets, const int64_t* ham_ids,
                                  double* const* out_values) {
    if (n_ctx < 0 || (n_ctx > 0 && (!ctxs || !batches || !plan_ids || !params || !param_offsets || !ham_ids || !out_values)))
        return fail(QB_ERR_INVALID, "null argument");
    for (int i = 0; i < n_ctx; ++i) {
        if (!ctxs[i]) return fail(QB_ERR_INVALID, "null context");
        for (int j = 0; j < i; ++j)
            if (ctxs[j] == ctxs[i]) return fail(QB_ERR_INVALID, "a context may appear once per call");
    }
    std::vector<Worker*> posted;
    for (int i = 0; i < n_ctx; ++i) {
        if (batches[i] <= 0) continue;
        qb_context* ctx = ctxs[i];
        {
            std::lock_guard<std::mutex> lock(ctx->worker_mu);
            if (!ctx->worker) {
                ctx->worker = std::make_unique<Worker>();
                Worker* w = ctx->worker.get();
                w->thread = std::thread([w] { w->loop(); });
            }
        }
        const int batch = batches[i];
        const int64_t* ids = plan_ids[i];
        const double* vals = params[i];
        const int64_t* offs = param_offsets[i];
        const int64_t ham = ham_ids[i];
        double* out = out_values[i];
        ctx->worker->post([=] { return qb_evaluate_expectation(ctx, batch, ids, vals, offs, ham, out); });
        posted.push_back(ctx->worker.get());
    }
    int rc = QB_OK;
    std::string first;
    for (Worker* w : posted) {  // wait for every device before reporting the first failure
        std::string msg;
        const int r = w->wait(msg);
        if (r != QB_OK && rc == QB_OK) rc = r, first = msg;
    }
    return rc == QB_OK ? QB_OK : fail(rc, first);
}

int qb_context_sm_count(qb_context* ctx) { return ctx ? ctx->sm_count : 0; }

uint64_t qb_context_workspace(qb_context* ctx) { return ctx ? workspace_limit_of(ctx) : 0; }

// ---- device memory / peer mapping for sharded states --------------------------------------------------
int qb_device_alloc(qb_context* ctx, uint64_t bytes, void** out_ptr) {
    if (!ctx || !out_ptr || !bytes) return fail(QB_ERR_INVALID, "null argument / zero size");
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, size_t(bytes));
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(QB_ERR_MEMORY, "cudaMalloc of " + std::to_string(bytes) + " bytes failed: " + cudaGetErrorString(e));
    }
    *out_ptr = p;
    return QB_OK;
}

int qb_device_free(qb_context* ctx, void* ptr) {
    if (!ctx) return fail(QB_ERR_INVALID, "null context");
    if (!ptr) return QB_OK;
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    QB_CUDA(cudaStreamSynchronize(ctx->stream));
    QB_CUDA(cudaFree(ptr));
    return QB_OK;
}

int qb_device_read(qb_context* ctx, const void* src, uint64_t offset, uint64_t bytes, void* host_out) {
    if (!ctx || !src || !host_out) return fail(QB_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    QB_CUDA(cudaMemcpyAsync(host_out, static_cast<const unsigned char*>(src) + offset, size_t(bytes), cudaMemcpyDeviceToHost, ctx->stream));
    QB_CUDA(cudaStreamSynchronize(ctx->stream));
    return QB_OK;
}

int qb_enable_peer_access(qb_context* ctx, int peer_device) {
    if (!ctx) return fail(QB_ERR_INVALID, "null context");
    if (peer_device == ctx->device) return QB_OK;
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    int can = 0;
    QB_CUDA(cudaDeviceCanAccessPeer(&can, ctx->device, peer_device));
    if (!can) return fail(QB_ERR_CUDA, "device " + std::to_string(ctx->device) + " cannot map the memory of device " + std::to_string(peer_device) + " (no peer access)");
    cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) {
        cudaGetLastError();
        return QB_OK;
    }
    if (e != cudaSuccess) return fail(QB_ERR_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
    return QB_OK;
}

static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handles are 64 bytes");

int qb_ipc_export(qb_context* ctx, void* ptr, unsigned char handle_out[64]) {
    if (!ctx || !ptr || !handle_out) return fail(QB_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    cudaIpcMemHandle_t h;
    QB_CUDA(cudaIpcGetMemHandle(&h, ptr));
    std::memcpy(handle_out, &h, 64);
    return QB_OK;
}

int qb_ipc_open(qb_context* ctx, const unsigned char handle[64], void** out_ptr) {
    if (!ctx || !handle || !out_ptr) return fail(QB_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, 64);
    void* p = nullptr;
    QB_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    *out_ptr = p;
    return QB_OK;
}

int qb_ipc_close(qb_context* ctx, void* mapped_ptr) {
    if (!ctx) return fail(QB_ERR_INVALID, "null context");
    if (!mapped_ptr) return QB_OK;
    std::lock_guard<std::mutex> lock(ctx->mu);
    QB_ON_DEVICE(ctx);
    QB_CUDA(cudaIpcCloseMemHandle(mapped_ptr));
    return QB_OK;
}

}  // extern "C"
