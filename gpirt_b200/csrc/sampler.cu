// The resident GP-IRT Gibbs sampler: device state + one sweep = the reference's loop body
// (src/gpirtMCMC.cpp:68-78 / :87-97) as a fixed sequence of kernel launches on one stream, and gpirt_b200_mcmc(),
// the drop-in for gpirtMCMC() (src/gpirtMCMC.cpp:5-117).
#include <sys/mman.h>

#include <cstdarg>
#include <cmath>
#include <algorithm>
#include <atomic>
#include <cstring>
#include <ctime>
#include <condition_variable>
#include <deque>
#include <functional>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include "comm.cuh"
#include "gemm_f64.cuh"
#include "kernels.cuh"
#include "linalg.cuh"
#include "ppc.cuh"
#include <climits>

#include "theta_int8.cuh"
#include "dgemm_i8.cuh"

namespace gpirt {

std::atomic<int64_t> g_launch_count{0};
thread_local int g_launch_priority_override = INT_MIN;
std::mutex& device_once_mutex() { static std::mutex mu; return mu; }
static thread_local char g_last_error[512] = "";
void set_last_error(const char* fmt, ...) {
    va_list ap; va_start(ap, fmt); vsnprintf(g_last_error, sizeof(g_last_error), fmt, ap); va_end(ap);
}
const char* last_error() { return g_last_error; }

int pool_alloc(void** p, size_t bytes, cudaStream_t st) {
    static bool configured[64] = {false};
    {
        DeviceOnce once(configured);
        int dev = 0;
        cudaMemPool_t pool;
        if (once.first && cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
            uint64_t keep = UINT64_MAX;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
    }
    cudaError_t e = cudaMallocAsync(p, bytes ? bytes : 256, st);
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_last_error("device allocation of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
        return GPIRT_B200_ERR_NOMEM;
    }
    return GPIRT_B200_OK;
}
void pool_free(void* p, cudaStream_t st) { if (p) cudaFreeAsync(p, st); }

// Host -> device copy of a large PAGEABLE array (the response matrix as R hands it over).  A plain cudaMemcpy of pageable
// memory is staged by the driver through one thread (~12 GB/s: 27 ms for the 328 MB of y at C3 — most of the cost of
// creating a sampler).  Here a few host threads copy 32 MiB pieces into two pinned slots and the DMA of one piece runs
// under the host copy of the next: the transfer then runs at the PCIe rate (~7 ms).
int upload_pageable(void* dst_dev, const void* src_host, size_t bytes, cudaStream_t st) {
    constexpr size_t PIECE = (size_t)32 << 20;
    static std::mutex mu;
    static void* slot[2] = {nullptr, nullptr};
    static cudaEvent_t ev[2] = {nullptr, nullptr};
    static bool recorded[2] = {false, false};
    static bool failed = false;                       // no pinned memory: plain copies from then on
    static int ev_device = -1;                        // the events belong to the device that was current when they were created
    std::lock_guard<std::mutex> lock(mu);
    int dev = 0;
    GP_CUDA(cudaGetDevice(&dev));
    if (bytes >= 2 * PIECE && !failed && !slot[0]) {
        ev_device = dev;
        for (int i = 0; i < 2 && !failed; ++i) {
            if (cudaHostAlloc(&slot[i], PIECE, cudaHostAllocDefault) != cudaSuccess || cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming) != cudaSuccess) {
                cudaGetLastError();
                failed = true;
            }
        }
        if (failed) { for (int i = 0; i < 2; ++i) { if (slot[i]) cudaFreeHost(slot[i]); slot[i] = nullptr; } }
    }
    if (bytes < 2 * PIECE || failed || !slot[1] || dev != ev_device) {
        GP_CUDA(cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, st));
        return GPIRT_B200_OK;
    }
    const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
    const int T = (int)std::min(12u, std::max(1u, hw * 3 / 4));
    const char* src = static_cast<const char*>(src_host);
    char* dst = static_cast<char*>(dst_dev);
    int k = 0;
    for (size_t off = 0; off < bytes; off += PIECE, ++k) {
        const int b = k & 1;
        const size_t len = std::min(PIECE, bytes - off);
        if (recorded[b]) GP_CUDA(cudaEventSynchronize(ev[b]));   // the DMA that last read this slot (possibly of an earlier call)
        {
            char* to = static_cast<char*>(slot[b]);
            const size_t per = (len / T + 4095) & ~(size_t)4095;
            std::vector<std::thread> th;
            for (int t = 1; t < T; ++t) {
                const size_t o = (size_t)t * per;
                if (o < len) th.emplace_back([=] { std::memcpy(to + o, src + off + o, std::min(per, len - o)); });
            }
            std::memcpy(to, src + off, std::min(per, len));
            for (auto& x : th) x.join();
        }
        GP_CUDA(cudaMemcpyAsync(dst + off, slot[b], len, cudaMemcpyHostToDevice, st));
        GP_CUDA(cudaEventRecord(ev[b], st));
        recorded[b] = true;
    }
    return GPIRT_B200_OK;
}

}  // namespace gpirt

using namespace gpirt;

// GPIRT_TRACE inside a captured sweep: CUDA events cannot be timed there, so the segment boundaries are tiny kernels that
// store %globaltimer (ns) — they replay with the graph, and the last replay's stamps are written out with the trace
__global__ void k_stamp(unsigned long long* slot) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    *slot = t;
}

// set around gpirt_b200_sampler_create by a several-chain call: chains after the first ignore GPIRT_TRACE
static thread_local bool t_untraced_create = false;

struct gpirt_b200_sampler {
    int n = 0, m = 0;
    int64_t ldn = 0, ldN = 0;       // leading dimensions (rounded up to 8 doubles) of n-row and 1001-row matrices
    gpirt_b200_opts opts{};
    RngKey key{};
    uint32_t item_offset = 0;
    Comm comm;
    cudaStream_t stream = nullptr;
    CholLookahead lookahead;
    ThetaInt8 ti8;               // tcgen05 int8 path of the theta contraction (no missing data)
    bool use_ti8 = false;
    // the two big FP64 products (nu = L Z, f* = A^T f) in 56-bit fixed point on the int8 tensor cores (dgemm_i8.cu):
    // digit planes of L, of A = S^-1 K* and of the item-side operand (Z before the ESS, f after it: never both alive)
    DigitPlanes dp_L, dp_A, dp_B;
    DigitPlanes dp_Linv, dp_LinvT, dp_K;   // L^-1 by rows, by columns (= rows of L^-T), and this rank's K* / L^-1 K* columns
    bool use_i8gemm = false;
    int lz_group = 4;            // finished Cholesky panels per slice of the pipelined L Z product
    // sweep pipelining: the latency-bound Cholesky chain of sweep t overlaps (a) the beta step of sweep t, (b) the Philox
    // fill of Z for sweep t+1 and (c) the product nu = L Z of sweep t+1, accumulated block column by block column behind
    // the factorisation (each group of lz_group finished panels contributes nu[r0:, :] += L[r0:, r0:r1] Z[r0:r1, :])
    bool pipeline = true;
    cudaStream_t st_beta = nullptr, st_lz = nullptr;
    cudaEvent_t ev_theta = nullptr, ev_z = nullptr, ev_beta = nullptr, ev_lz = nullptr;
    cudaEvent_t ev_linv = nullptr, ev_solve = nullptr, ev_fwd = nullptr;
    // What a pipelined sweep leaves for the next one.  The K* solves of the NEXT sweep depend on theta and the factor
    // only: rebuild_pipelined leaves them pending and the next sweep starts them on a side stream right before its ESS,
    // so that they run beside it — and so that every side stream is joined at the end of a sweep, which is what lets the
    // whole pipelined sweep be captured as a CUDA graph.
    struct Carry {
        enum class Start { NONE, BWD, LINV_SOLVES };   // backward substitution of this rank's grid columns (the forward
                                                       // steps trailed the panels), or the solves through L^-1
        enum class Solved { NONE, LOCAL, ALL };        // in flight behind ev_solve: this rank's slice of S^-1 K* and s (not
                                                       // yet gathered), or S^-1 K* and s complete for the current theta
        bool nu_ready = false;       // nu already holds L z for sweep nu_sweep
        uint32_t nu_sweep = 0;
        Start start = Start::NONE;   // K* work the next sweep starts before its ESS
        Solved solved = Solved::NONE;
        bool ess_yields = false;     // the backward pass was just started: the ESS that follows must leave it SMs
    } carry;
    // discards the carried state (the sampler's state was changed from outside the sweep, or the sweep's shape changes)
    void drop_carry() {
        if (carry.solved != Carry::Solved::NONE) cudaStreamWaitEvent(stream, ev_solve, 0);
        carry = Carry{};
    }
    int prio_second = 0;            // one notch below the top stream priority
    int launch_deferred_solves();
    int fstar_solves(cudaStream_t st);
    // Route of the K* solves, chosen once in create():
    //   LINV     (default on one GPU for n <= 6144) through L^-1
    //   SUBST    (default with items sharded over GPUs, and for n > 6144) the two triangular solves for this rank's slice
    //            of the grid columns as blocked substitutions with the 128-block inverses of the factorisation — no L^-1.
    //            The forward steps trail the Cholesky panels on st_trsm; only the backward pass (32 short steps) follows
    //            the factorisation.  With few right-hand sides per rank this replaces the replicated 1.3 ms L^-1 +
    //            products by a ~0.4 ms chain.
    //   LITERAL  opts.fstar_mode = 1: the reference's per-item solves, through L^-1
    enum class Route { LINV, SUBST, LITERAL } route = Route::LINV;
    cudaStream_t st_trsm = nullptr;
    void grid_slice(int& c0, int& nc) const {
        const int per = (int)ceil_div(N_GRID, comm.world);
        c0 = std::min(N_GRID, comm.rank * per);
        nc = std::min(N_GRID, c0 + per) - c0;
    }
    int trsm_kstar(cudaStream_t st);
    int trsm_fwd_step(cudaStream_t st, int k);
    int trsm_bwd(cudaStream_t st, bool leading_blocks_inverted = false);
    int bwd_block() const;                 // order of the diagonal-block inverses the backward substitution runs on
    int invert_bwd_step(cudaStream_t st, int k);
    double* splitk_ws = nullptr;           // partial tiles of the split-K products of the backward pass (thin: few grid columns per rank)
    int* splitk_count = nullptr;
    GemmArgs thin(GemmArgs a) const;
    int gather_solves(cudaStream_t st);
    bool has_missing = false;
    int ess_shape = -1, beta_shape = -1;   // ItemShape the last ESS / beta launch picked (gpirt_b200_sampler_uses)
    bool timing = true;
    uint32_t sweep_counter = 0;
    int64_t launches_at_create = 0;

    int8_t* y8 = nullptr; int64_t ldy8 = 0;
    double *yd = nullptr, *theta = nullptr, *theta_star = nullptr, *prior = nullptr, *beta = nullptr, *pm = nullptr,
           *psd = nullptr, *pstep = nullptr, *L = nullptr, *Dinv = nullptr, *f = nullptr, *Z = nullptr, *nu = nullptr,
           *fstar = nullptr, *Dmat = nullptr, *irf_sum = nullptr, *kstar = nullptr, *s = nullptr, *logPt = nullptr,
           *partial = nullptr, *Linv = nullptr, *Tmp = nullptr, *kstar2 = nullptr;
    int* work = nullptr;   // item counters of the persistent per-item kernels: [0] ESS, [1] beta
    int* chol_flags = nullptr;   // scratch of the factorisation: one counter per panel step
    int *nprop = nullptr, *theta_idx = nullptr, *status = nullptr;  // status[0] chol, [1] ess, [2] theta-degenerate count
    unsigned long long* counters = nullptr;                        // [0] missing cells, [1] illegal cells
    static constexpr int N_CHUNKS = 128;   // item chunks of the D row sums: enough CTAs to cover the HBM latency of the column walk

    // ---- timers ----
    struct Seg { int timer; cudaEvent_t a, b; int slot = -1; };
    unsigned long long* d_stamps = nullptr;       // 2 slots per traced segment of the captured sweep
    std::vector<std::pair<int, int>> stamp_segs;  // (timer, first slot)
    static constexpr int MAX_STAMPS = 4096;
    bool stamping() const { return trace_file && capturing && d_stamps && (int)stamp_segs.size() * 2 + 2 <= MAX_STAMPS; }
    void dump_stamps() {
        if (!trace_file || !d_stamps || stamp_segs.empty()) return;
        std::vector<unsigned long long> h(2 * stamp_segs.size());
        if (cudaMemcpy(h.data(), d_stamps, h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost) != cudaSuccess) return;
        unsigned long long t0 = ~0ull;
        for (auto v : h) if (v && v < t0) t0 = v;
        fprintf(trace_file, "# graph sweep (last replay) %d x %d\n", n, m);
        for (auto& sg : stamp_segs) {
            const unsigned long long a = h[sg.second], b = h[sg.second + 1];
            if (a && b) fprintf(trace_file, "%d %.4f %.4f\n", sg.first, (a - t0) * 1e-6, (b - t0) * 1e-6);
        }
        fflush(trace_file);
    }
    std::vector<Seg> pending;
    std::vector<cudaEvent_t> pool;
    double ms[GPIRT_B200_TIMER_COUNT] = {0};
    int64_t calls[GPIRT_B200_TIMER_COUNT] = {0};
    Seg cur{};

    Seg tic_on(int timer, cudaStream_t st) {
        Seg sg{timer, nullptr, nullptr};
        if (stamping()) {
            sg.slot = 2 * (int)stamp_segs.size();
            stamp_segs.push_back({timer, sg.slot});
            k_stamp<<<1, 1, 0, st>>>(d_stamps + sg.slot);
            return sg;
        }
        if (!timing || capturing) return sg;
        sg.a = get_event(); sg.b = get_event();
        cudaEventRecord(sg.a, st);
        return sg;
    }
    void toc_on(Seg& sg, cudaStream_t st) {
        if (sg.slot >= 0) { k_stamp<<<1, 1, 0, st>>>(d_stamps + sg.slot + 1); return; }
        if (!timing || !sg.a) return;
        cudaEventRecord(sg.b, st);
        pending.push_back(sg);
    }

    cudaEvent_t get_event() {
        if (!pool.empty()) { cudaEvent_t e = pool.back(); pool.pop_back(); return e; }
        cudaEvent_t e; cudaEventCreate(&e); return e;
    }
    void tic(int timer) { cur = tic_on(timer, stream); }
    void toc() { toc_on(cur, stream); }
    // GPIRT_TRACE=<file>: every timed segment is also written as "timer start_ms end_ms" relative to the sampler's
    // creation (segments of different streams overlap: this is the timeline the per-timer sums cannot show)
    cudaEvent_t trace_ref = nullptr;
    FILE* trace_file = nullptr;
    void flush_timers() {  // call after ALL of the sampler's streams have been synchronised
        for (auto& sg : pending) {
            float t = 0.f;
            if (cudaEventElapsedTime(&t, sg.a, sg.b) == cudaSuccess) { ms[sg.timer] += t; calls[sg.timer] += 1; }
            if (trace_file && trace_ref) {
                float t0 = 0.f, t1 = 0.f;
                if (cudaEventElapsedTime(&t0, trace_ref, sg.a) == cudaSuccess && cudaEventElapsedTime(&t1, trace_ref, sg.b) == cudaSuccess)
                    fprintf(trace_file, "%d %.4f %.4f\n", sg.timer, t0, t1);
            }
            pool.push_back(sg.a); pool.push_back(sg.b);
        }
        pending.clear();
        cudaGetLastError();   // a not-ready event must not surface later as a launch failure
    }

    // while a sweep is being captured into a graph the kernels get the sweep counter relative to the captured sweep plus
    // the device word the graph bumps on every replay
    RngKey key_at(uint32_t sweep) const {
        RngKey k = key;
        k.sweep = capturing ? sweep - capture_base : sweep;
        k.sweep_dev = capturing ? d_sweep : nullptr;
        return k;
    }
    // ---- CUDA graph of a sweep (small n: ~20 short kernels, pure launch latency; n > 256: the pipelined sweep, whose
    // Cholesky chain takes ~15 host API calls per panel — with items sharded the host is the limit otherwise) ----
    bool graph_enabled = true, capturing = false, warmed = false;   // graph_enabled: opts.use_graph >= 0 and capturable
    uint32_t capture_base = 0;
    uint32_t* d_sweep = nullptr;          // device copy of the sweep counter read by the captured kernels
    uint32_t d_sweep_value = 0xffffffffu; // what *d_sweep holds (host mirror)
    cudaGraphExec_t gexec[2] = {nullptr, nullptr};   // [accumulate_irf]
    int64_t graph_replays = 0;            // sweeps run as a graph launch (gpirt_b200_sampler_uses(s, 5))
    Carry graph_carry[2];                 // what the captured sweep left, nu_sweep relative to the captured sweep
    void drop_graphs() { for (auto& g : gexec) if (g) { cudaGraphExecDestroy(g); g = nullptr; } }
    int64_t graph_kernels = 0;            // kernels per sweep (counted on the eager path; a graph replay launches the same ones)
    int sweep_eager(uint32_t t, int accumulate);
    int sweep_graph(uint32_t t, int accumulate);

    template <typename T> int alloc(T*& p, size_t count) {
        void* q = nullptr;
        GP_TRY(pool_alloc(&q, count * sizeof(T) + 256, stream));
        p = (T*)q;
        return GPIRT_B200_OK;
    }

    int create(const double* y, int64_t n_, int64_t m_, const double* theta_init, const double* pm_h, const double* psd_h,
               const double* pstep_h, const gpirt_b200_opts* o);
    int init_draws();
    int step_draw_f(uint32_t sweep);
    int step_draw_fstar(uint32_t sweep, int accumulate);
    int step_draw_theta(uint32_t sweep);
    int step_draw_beta(uint32_t sweep);
    int step_rebuild();
    int ess_only(uint32_t sweep);
    int rebuild_pipelined(uint32_t sweep, uint32_t next_sweep);
    int sweep(int accumulate);
    int check_status();
    void destroy();
};

static int upload_padded(double* dst, int64_t ld, const double* src_host, int rows, int cols, cudaStream_t st) {
    GP_CUDA(cudaMemcpy2DAsync(dst, ld * sizeof(double), src_host, (size_t)rows * sizeof(double), (size_t)rows * sizeof(double),
                              cols, cudaMemcpyHostToDevice, st));
    return GPIRT_B200_OK;
}
static int download_padded(double* dst_host, const double* src, int64_t ld, int rows, int cols, cudaStream_t st) {
    GP_CUDA(cudaMemcpy2DAsync(dst_host, (size_t)rows * sizeof(double), src, ld * sizeof(double), (size_t)rows * sizeof(double),
                              cols, cudaMemcpyDeviceToHost, st));
    return GPIRT_B200_OK;
}

int gpirt_b200_sampler::create(const double* y, int64_t n_, int64_t m_, const double* theta_init, const double* pm_h,
                               const double* psd_h, const double* pstep_h, const gpirt_b200_opts* o) {
    if (!y || !theta_init || !pm_h || !psd_h || !pstep_h || n_ <= 0 || m_ <= 0 || n_ > (1 << 20) || m_ > (1 << 24)) {
        set_last_error("bad argument: null pointer or n, m out of range");
        return GPIRT_B200_ERR_ARG;
    }
    if (o) opts = *o;
    if (opts.world_size > 1) {   // item sharding: every rank can check these without talking to its peers
        if (opts.rank < 0 || opts.rank >= opts.world_size || opts.world_size > 4096) {
            set_last_error("bad argument: rank %d of world_size %d", opts.rank, opts.world_size);
            return GPIRT_B200_ERR_ARG;
        }
        if (opts.m_global < opts.world_size || opts.item_offset < 0 || opts.item_offset + m_ > opts.m_global) {
            set_last_error("bad argument: item block [%lld, %lld) of m_global = %lld on %d ranks (every rank needs at least one item)",
                           (long long)opts.item_offset, (long long)(opts.item_offset + m_), (long long)opts.m_global, opts.world_size);
            return GPIRT_B200_ERR_ARG;
        }
    }
    n = (int)n_; m = (int)m_;
    ldn = round_up(n, 8); ldN = round_up(N_GRID, 8); ldy8 = round_up(n, 16);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        set_last_error("no CUDA device available (this library has no CPU fallback)");
        return GPIRT_B200_ERR_CUDA;
    }
    if (o && opts.device >= 0) GP_CUDA(cudaSetDevice(opts.device));
    key.k0 = (uint32_t)opts.seed; key.k1 = (uint32_t)(opts.seed >> 32); key.sweep = 0; key.sweep_dev = nullptr;
    graph_enabled = opts.use_graph >= 0;
    if (opts.world_size > 1) {
        item_offset = (uint32_t)opts.item_offset;
        GP_TRY(comm_init(comm, opts.rank, opts.world_size, opts.nccl_unique_id));
    }
    launches_at_create = g_launch_count;
    if (const char* tf = t_untraced_create ? nullptr : getenv("GPIRT_TRACE")) {
        if (opts.rank == 0 || opts.world_size <= 1) trace_file = fopen(tf, "a");
        if (trace_file) fprintf(trace_file, "# sampler %d x %d world %d\n", n, m, opts.world_size > 1 ? opts.world_size : 1);
    }
    {   // the factorisation chain and its bulk updates run at the highest priority, the overlapped L Z product at the lowest
        int least = 0, greatest = 0;
        GP_CUDA(cudaDeviceGetStreamPriorityRange(&least, &greatest));
        GP_CUDA(cudaStreamCreateWithPriority(&stream, cudaStreamNonBlocking, greatest));
        GP_CUDA(cudaStreamCreateWithPriority(&lookahead.aux, cudaStreamNonBlocking, greatest));
        GP_CUDA(cudaStreamCreateWithPriority(&st_beta, cudaStreamNonBlocking, least));
        GP_CUDA(cudaStreamCreateWithPriority(&st_lz, cudaStreamNonBlocking, least));
        prio_second = greatest < least ? greatest + 1 : greatest;
        // the substitution steps that trail the panels yield to the chain itself
        GP_CUDA(cudaStreamCreateWithPriority(&st_trsm, cudaStreamNonBlocking, greatest < least ? greatest + 1 : greatest));
        for (cudaEvent_t* e : {&ev_theta, &ev_z, &ev_beta, &ev_lz, &ev_linv, &ev_solve, &ev_fwd}) GP_CUDA(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
        if (trace_file) {
            GP_CUDA(cudaEventCreate(&trace_ref)); GP_CUDA(cudaEventRecord(trace_ref, stream));
            GP_CUDA(cudaMalloc((void**)&d_stamps, MAX_STAMPS * sizeof(unsigned long long)));
            GP_CUDA(cudaMemset(d_stamps, 0, MAX_STAMPS * sizeof(unsigned long long)));
        }
        // GPIRT_SOLVE_MODE = 0 / 1 forces the route through L^-1 / by substitution.  Through L^-1 costs n^3/3 for the
        // inverse + two triangular products, blocked substitution behind the Cholesky panels 2 n^2 x 1001: substitution
        // wins when few right-hand sides are left per rank, and on one GPU once n/3 > 2 x 1001
        const char* sm = getenv("GPIRT_SOLVE_MODE");
        const bool subst = sm ? atoi(sm) == 1 : (comm.world > 1 || n > 6144);
        if (opts.fstar_mode != 0) route = Route::LITERAL;   // the literal per-item form needs L^-1
        else route = subst ? Route::SUBST : Route::LINV;
    }

    const size_t nm = (size_t)ldn * m, Nm = (size_t)ldN * m;
    // K* / S^-1 K* hold world x ceil(1001 / world) grid columns: the in-place all-gather of the per-rank slices pads the
    // last rank's slice to full width
    const size_t kcols = (size_t)comm.world * (size_t)ceil_div(N_GRID, comm.world) + 8;
    {   // the theta contraction runs on the int8 tensor cores (y is an exact int8 operand); GPIRT_THETA_INT8=0 keeps
        // the FP64 DMMA contraction instead, which needs y as doubles
        const char* e = getenv("GPIRT_THETA_INT8");
        use_ti8 = e ? atoi(e) != 0 : true;
    }
    GP_TRY(alloc(y8, (size_t)ldy8 * m));
    if (!use_ti8) GP_TRY(alloc(yd, nm));
    GP_TRY(alloc(theta, (size_t)ldn)); GP_TRY(alloc(theta_star, (size_t)ldN)); GP_TRY(alloc(prior, (size_t)ldN));
    GP_TRY(alloc(beta, 2 * (size_t)m)); GP_TRY(alloc(pm, 2 * (size_t)m)); GP_TRY(alloc(psd, 2 * (size_t)m)); GP_TRY(alloc(pstep, 2 * (size_t)m));
    GP_TRY(alloc(L, (size_t)ldn * n)); GP_TRY(alloc(Dinv, (size_t)ldn * CHOL_NB));
    GP_TRY(alloc(Linv, (size_t)ldn * n)); GP_TRY(alloc(Tmp, (size_t)ldn * n)); GP_TRY(alloc(kstar2, (size_t)ldn * kcols));
    GP_TRY(alloc(chol_flags, (size_t)ceil_div(n, CHOL_NB) + 1));
    GP_TRY(alloc(f, nm)); GP_TRY(alloc(Z, nm)); GP_TRY(alloc(nu, nm));
    GP_TRY(alloc(fstar, Nm)); GP_TRY(alloc(Dmat, Nm)); GP_TRY(alloc(irf_sum, Nm));
    GP_TRY(alloc(kstar, (size_t)ldn * kcols)); GP_TRY(alloc(s, std::max((size_t)ldN, kcols)));
    if (route == Route::SUBST) {
        // split-K workspace: the thin products of the backward pass (M <= 4096 rows x this rank's grid columns, 8 splits) and
        // the batched late levels of the block inverses (n / 1024 pairs of 512 x 512 tiles, 4 splits)
        const size_t per = (size_t)ceil_div(N_GRID, comm.world);
        const size_t ws_doubles = std::max((size_t)round_up(std::min(n, 4096), 128) * (size_t)round_up((int64_t)per, 128) * 8, (size_t)n * 1024);
        const size_t ws_tiles = std::max((size_t)ceil_div(std::min(n, 4096), 64) * (size_t)ceil_div((int64_t)per, 64), (size_t)n / 8) + 64;
        GP_TRY(alloc(splitk_ws, ws_doubles));
        GP_TRY(alloc(splitk_count, ws_tiles));
        GP_CUDA(cudaMemsetAsync(splitk_count, 0, ws_tiles * sizeof(int), stream));
        GP_CUDA(cudaMemsetAsync(Linv, 0, (size_t)ldn * n * sizeof(double), stream));   // block inverses: only their lower parts are rewritten
    }
    GP_TRY(alloc(logPt, (size_t)ldN * (n + 1))); GP_TRY(alloc(partial, (size_t)N_CHUNKS * N_GRID));
    GP_TRY(alloc(nprop, (size_t)m)); GP_TRY(alloc(theta_idx, (size_t)n)); GP_TRY(alloc(status, 4)); GP_TRY(alloc(counters, 2)); GP_TRY(alloc(work, 4));
    GP_TRY(alloc(d_sweep, 2));
    GP_CUDA(cudaMemsetAsync(status, 0, 4 * sizeof(int), stream));
    GP_CUDA(cudaMemsetAsync(Dinv, 0, (size_t)ldn * CHOL_NB * sizeof(double), stream));   // the factorisation writes the lower triangles only
    GP_CUDA(cudaMemsetAsync(counters, 0, 2 * sizeof(unsigned long long), stream));
    GP_CUDA(cudaMemsetAsync(irf_sum, 0, Nm * sizeof(double), stream));
    GP_CUDA(cudaMemsetAsync(y8, 0, (size_t)ldy8 * m, stream));
    if (yd) GP_CUDA(cudaMemsetAsync(yd, 0, nm * sizeof(double), stream));
    GP_CUDA(cudaMemsetAsync(f, 0, nm * sizeof(double), stream));
    GP_CUDA(cudaMemsetAsync(fstar, 0, Nm * sizeof(double), stream));
    GP_CUDA(cudaMemsetAsync(logPt, 0, (size_t)ldN * (n + 1) * sizeof(double), stream));
    GP_CUDA(cudaMemsetAsync(nprop, 0, (size_t)m * sizeof(int), stream));
    GP_CUDA(cudaMemsetAsync(theta_idx, 0, (size_t)n * sizeof(int), stream));

    // y arrives as R hands it over: REALSXP n x m, {1,-1,NA}; staged through the nu buffer (tight n x m fits in ldn x m)
    GP_TRY(upload_pageable(nu, y, (size_t)n * m * sizeof(double), stream));
    GP_TRY(launch_ingest_y(stream, nu, n, m, y8, ldy8, yd, ldn, counters, counters + 1));
    unsigned long long cnt[2];
    GP_CUDA(cudaMemcpyAsync(cnt, counters, sizeof(cnt), cudaMemcpyDeviceToHost, stream));
    GP_CUDA(cudaMemcpyAsync(theta, theta_init, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, stream));
    GP_CUDA(cudaMemcpyAsync(pm, pm_h, 2 * (size_t)m * sizeof(double), cudaMemcpyHostToDevice, stream));
    GP_CUDA(cudaMemcpyAsync(psd, psd_h, 2 * (size_t)m * sizeof(double), cudaMemcpyHostToDevice, stream));
    GP_CUDA(cudaMemcpyAsync(pstep, pstep_h, 2 * (size_t)m * sizeof(double), cudaMemcpyHostToDevice, stream));
    GP_TRY(launch_grid_init(stream, theta_star, prior));
    GP_CUDA(cudaStreamSynchronize(stream));
    if (cnt[1] != 0) {
        set_last_error("y holds %llu values that are not +1, -1 or NA", cnt[1]);
        return GPIRT_B200_ERR_Y_VALUE;
    }
    has_missing = cnt[0] != 0;
    if (use_ti8) GP_TRY(ti8.init(stream, y8, ldy8, n, m, has_missing));
    {   // GPIRT_GEMM_INT8 = 1 / 0 forces the fixed-point tensor-core products on / off (FP64 DMMA instead)
        const char* e = getenv("GPIRT_GEMM_INT8");
        use_i8gemm = e ? atoi(e) != 0 : (n >= 512 && std::max<int64_t>(m, opts.m_global) >= 256);   // same path on every shard
        if (n >= 65536) use_i8gemm = false;   // int32 accumulators hold 8 x 64 x 64 x K
        if (use_i8gemm) {
            GP_TRY(dp_L.init(stream, n, n, 128));
            GP_TRY(dp_A.init(stream, N_GRID, n, 128));
            GP_TRY(dp_B.init(stream, m, n, 64));
            if (route == Route::LINV) {
                int c0, nc;
                grid_slice(c0, nc);
                GP_TRY(dp_Linv.init(stream, n, n, 128));
                GP_TRY(dp_LinvT.init(stream, n, n, 128));
                if (nc > 0) GP_TRY(dp_K.init(stream, nc, n, 64));
            }
            lz_group = 16;
        }
    }
    GP_TRY(step_rebuild());                                                         // gpirtMCMC.cpp:15-17
    GP_CUDA(cudaStreamSynchronize(stream));
    return check_status();
}

int gpirt_b200_sampler::check_status() {
    int h[4];
    GP_CUDA(cudaMemcpyAsync(h, status, sizeof(h), cudaMemcpyDeviceToHost, stream));
    GP_CUDA(cudaStreamSynchronize(stream));
    if (st_lz) GP_CUDA(cudaStreamSynchronize(st_lz));       // side streams may still run the next sweep's K* solves
    if (st_beta) GP_CUDA(cudaStreamSynchronize(st_beta));
    if (st_trsm) GP_CUDA(cudaStreamSynchronize(st_trsm));
    flush_timers();
    if (h[0]) { set_last_error("chol(): decomposition failed"); return GPIRT_B200_ERR_NOT_PD; }
    if (h[1]) { set_last_error("elliptical slice sampler did not terminate (NaN log-likelihood?)"); return GPIRT_B200_ERR_ESS; }
    return GPIRT_B200_OK;
}

// S = K(theta,theta); S.diag() += 0.001; cholS = chol(S,"lower")                     gpirtMCMC.cpp:76-78
int gpirt_b200_sampler::step_rebuild() {
    tic(GPIRT_B200_T_KBUILD);
    GP_TRY(launch_se_cov(stream, theta, n, theta, n, 0.001, true, L, ldn));
    toc();
    tic(GPIRT_B200_T_CHOL);
    GP_TRY(potrf_lower_rl(stream, L, ldn, n, Dinv, ldn, status, chol_flags, &lookahead));
    toc();
    if (route != Route::SUBST) {
        tic(GPIRT_B200_T_TRTRI);   // L^-1 once per sweep: every triangular solve of draw_fstar becomes a triangular GEMM
        GP_TRY(trtri_lower(stream, L, ldn, n, Dinv, ldn, Linv, ldn, Tmp, ldn));
        toc();
    }
    return GPIRT_B200_OK;
}

// |L_ik| <= sqrt(K_ii) = sqrt(1.001) < 2: one fixed scale for every row of L, so L can be sliced while later panels of
// the factorisation are still running
constexpr int L_FIXED_EXP = 1;
constexpr int LZ_GROUP_COLS = 24, FSTAR_GROUP_COLS = 18;   // column tiles per L2-resident group (dgemm_i8)

static GemmArgs G(int M, int N, int K, const double* A, int64_t lda, const double* B, int64_t ldb, double* C, int64_t ldc,
                  double alpha, double beta, int tri, int b_abs = 0) {
    GemmArgs g;
    g.M = M; g.N = N; g.K = K; g.A = A; g.lda = lda; g.B = B; g.ldb = ldb; g.C = C; g.ldc = ldc;
    g.alpha = alpha; g.beta = beta; g.tri = tri; g.b_abs = b_abs;
    return g;
}

// f = draw_f(f, y, cholS, mu)                                                       gpirtMCMC.cpp:68, draw-f.cpp:64-73
int gpirt_b200_sampler::step_draw_f(uint32_t sweep) {
    const RngKey k = key_at(sweep);
    tic(GPIRT_B200_T_FILL_Z);
    if (use_i8gemm)   // the normals go straight into the digit planes of the product's operand
        GP_TRY(launch_fill_normal_planes(stream, dp_B.planes, dp_B.scale, dp_B.rows_pad, dp_B.k_pad, n, m, k,
                                         sweep == 0 ? P_INIT_F_Z : P_ESS_Z, item_offset, nullptr, ldn));
    else GP_TRY(launch_fill_normal(stream, Z, n, m, ldn, k, sweep == 0 ? P_INIT_F_Z : P_ESS_Z, item_offset));
    toc();
    tic(GPIRT_B200_T_LZ_GEMM);   // nu_j = cholS z_j for all items in one product (mvnormal.h:10)
    if (use_i8gemm) {
        GP_TRY(dp_L.slice_mcontig(stream, L, ldn, true, 0, n, L_FIXED_EXP));
        GP_TRY(dgemm_i8(stream, dp_L, dp_B, sweep == 0 ? f : nu, ldn, DG_TRI_LOWER, 0, n, false, LZ_GROUP_COLS));
    } else {
        GP_TRY(gemm_f64(stream, false, false, G(n, m, n, L, ldn, Z, ldn, sweep == 0 ? f : nu, ldn, 1.0, 0.0, TRI_A_LOWER)));
    }
    toc();
    if (sweep == 0) return GPIRT_B200_OK;   // initial f_j = rmvnorm(cholS), gpirtMCMC.cpp:19-21
    tic(GPIRT_B200_T_ESS);
    GP_TRY(launch_ess(stream, f, nu, ldn, y8, ldy8, theta, beta, n, m, k, item_offset, nprop, status + 1, work, &ess_shape));
    toc();
    return GPIRT_B200_OK;
}

// The item-independent part of draw_fstar (draw-fstar.cpp:17-20): kstar = K(theta, theta*), tmp = L^-1 kstar,
// s = 1 - sqrt(colsum(tmp % tmp)), and A = L^-T tmp so that K*^T L^-T L^-1 f_j = A^T f_j needs one product per sweep
// instead of two solves per item.  Depends on theta and L only, so the pipelined sweep runs it beside the ESS.
int gpirt_b200_sampler::trsm_kstar(cudaStream_t st) {   // K(theta, theta*) for this rank's grid columns      :17
    int c0, nc;
    grid_slice(c0, nc);
    if (nc > 0) GP_TRY(launch_se_cov(st, theta, n, theta_star + c0, nc, 0.0, false, kstar + (int64_t)c0 * ldn, ldn));
    return GPIRT_B200_OK;
}
// forward substitution, block row k:  X_k = L_kk^-1 B_k,  B[below] -= L[below, k] X_k   (B = kstar, X = kstar2)     :19
int gpirt_b200_sampler::trsm_fwd_step(cudaStream_t st, int k) {
    int c0, nc;
    grid_slice(c0, nc);
    if (nc <= 0) return GPIRT_B200_OK;
    const int r0 = k * CHOL_NB, nb = std::min(CHOL_NB, n - r0), rem = n - r0 - nb;
    double* B = kstar + (int64_t)c0 * ldn;
    double* X = kstar2 + (int64_t)c0 * ldn;
    GP_TRY(gemm_f64(st, false, false, G(nb, nc, nb, Dinv + r0, ldn, B + r0, ldn, X + r0, ldn, 1.0, 0.0, TRI_A_LOWER)));
    if (rem > 0)
        GP_TRY(gemm_f64(st, false, false, G(rem, nc, nb, L + (r0 + nb) + (int64_t)r0 * ldn, ldn, X + r0, ldn, B + r0 + nb, ldn, -1.0, 1.0, TRI_NONE)));
    return GPIRT_B200_OK;
}
// s from tmp = L^-1 K* (:20), then the backward substitution  L^T A = tmp  (tmp = kstar2 is consumed, A -> kstar)    :24
// The backward pass cannot trail the factorisation (it starts at the last block), so it is the serial tail of the sharded
// sweep: instead of 32 steps with the 128-blocks it runs with the inverses of 1024 x 1024 diagonal blocks (built from the
// 128-block inverses by three levels of batched recursive doubling) — 4 steps of two products each.  With a handful of
// grid columns per rank those products are thin (126 columns at 8 GPUs: 32 output tiles, K = 1024), so they are split
// over K (deterministic split-K, gemm_f64.cuh); and every diagonal-block inverse but the last is computed behind the
// factorisation (invert_bwd_block from the panel hook), which leaves one block inverse and seven short products in the tail.
int gpirt_b200_sampler::bwd_block() const { return n >= 2048 ? 1024 : (n >= 1024 ? 512 : CHOL_NB); }
// the split factor depends on the shape of the product's A operand only — never on the number of right-hand sides, i.e.
// on how many ranks share the grid columns: a sharded run stays bit-identical to the unsharded one
GemmArgs gpirt_b200_sampler::thin(GemmArgs a) const {
    if (splitk_ws && a.K >= 512 && a.M <= 4096) {
        a.splitk = (int)std::min<int64_t>(8, a.K / 128);
        a.ws = splitk_ws;
        a.ws_count = splitk_count;
    }
    return a;
}
// the inverses of the diagonal blocks of order bwd_block() grow on the diagonal of Linv behind the factorisation: step k
// (after panel k) adds the 128-block inverse of panel k and every merge that panel completes (trtri_lower_step)
int gpirt_b200_sampler::invert_bwd_step(cudaStream_t st, int k) {
    const int blk = bwd_block();
    if (blk <= CHOL_NB) return GPIRT_B200_OK;
    return trtri_lower_step(st, L, ldn, n, Dinv, ldn, Linv, ldn, Tmp, ldn, blk, k, splitk_ws, splitk_count);
}
int gpirt_b200_sampler::trsm_bwd(cudaStream_t st, bool leading_blocks_inverted) {
    int c0, nc;
    grid_slice(c0, nc);
    if (nc <= 0) return GPIRT_B200_OK;
    double* A = kstar + (int64_t)c0 * ldn;
    double* Y = kstar2 + (int64_t)c0 * ldn;
    GP_TRY(launch_fstar_sd(st, Y, ldn, n, nc, s + c0));
    const int blk = bwd_block();
    const int nblk = (int)ceil_div(n, blk);
    const double* Xb = Dinv;       // leaf inverses: block k at rows k * blk of an n x blk array ...
    int64_t ldx = ldn, diag_step = 0;
    if (blk > CHOL_NB) {           // ... or on the diagonal of Linv (n x n)
        Seg sg = tic_on(GPIRT_B200_T_TRTRI, st);
        if (leading_blocks_inverted) GP_TRY(invert_bwd_step(st, (int)ceil_div(n, CHOL_NB) - 1));   // only the merges the last panel completes
        else GP_TRY(trtri_lower(st, L, ldn, n, Dinv, ldn, Linv, ldn, Tmp, ldn, blk, splitk_ws, splitk_count));
        toc_on(sg, st);
        Xb = Linv; diag_step = ldn;
    }
    for (int k = nblk - 1; k >= 0; --k) {
        const int r0 = k * blk, nb = std::min(blk, n - r0);
        GP_TRY(gemm_f64(st, true, false, thin(G(nb, nc, nb, Xb + r0 + (int64_t)r0 * diag_step, ldx, Y + r0, ldn, A + r0, ldn, 1.0, 0.0, TRI_A_UPPER))));
        if (r0 > 0)
            GP_TRY(gemm_f64(st, true, false, thin(G(r0, nc, nb, L + r0, ldn, A + r0, ldn, Y, ldn, -1.0, 1.0, TRI_NONE))));
    }
    return GPIRT_B200_OK;
}
int gpirt_b200_sampler::gather_solves(cudaStream_t st) {
    if (comm.world > 1) {
        const int per = (int)ceil_div(N_GRID, comm.world);
        GP_TRY(comm_allgather_f64(comm, kstar, (size_t)per * ldn, st));
        GP_TRY(comm_allgather_f64(comm, s, (size_t)per, st));
    }
    if (use_i8gemm) GP_TRY(dp_A.slice_kcontig(st, kstar, ldn));   // row k of A^T = column k of S^-1 K*
    return GPIRT_B200_OK;
}

// With items sharded over GPUs this part would be replicated: instead every rank solves for its slice of the 1001 grid
// columns and the slices are all-gathered (n x 1001 doubles) — through L^-1 the caller passes the main stream then
int gpirt_b200_sampler::fstar_solves(cudaStream_t st) {
    Seg a = tic_on(GPIRT_B200_T_KSTAR, st);
    GP_TRY(trsm_kstar(st));
    toc_on(a, st);
    Seg b = tic_on(GPIRT_B200_T_TRSM, st);
    int c0, nc;
    grid_slice(c0, nc);
    double* Kc = kstar + (int64_t)c0 * ldn;
    double* K2c = kstar2 + (int64_t)c0 * ldn;
    if (route == Route::SUBST) {
        const int nblk = (int)ceil_div(n, CHOL_NB);
        for (int k = 0; k < nblk; ++k) GP_TRY(trsm_fwd_step(st, k));
        GP_TRY(trsm_bwd(st));
    } else if (nc > 0 && use_i8gemm) {
        // the two triangular products with L^-1 in fixed point as well (L^-1 has zeros above the diagonal: trtri_lower)
        GP_TRY(dp_Linv.slice_mcontig(st, Linv, ldn, true, 0, n, INT_MIN));
        GP_TRY(dp_LinvT.slice_kcontig(st, Linv, ldn));
        GP_TRY(dp_K.slice_kcontig(st, Kc, ldn));
        GP_TRY(dgemm_i8(st, dp_Linv, dp_K, K2c, ldn, DG_TRI_LOWER, 0, n, false, 0));      // :19
        GP_TRY(launch_fstar_sd(st, K2c, ldn, n, nc, s + c0));                             // :20
        GP_TRY(dp_K.slice_kcontig(st, K2c, ldn));
        GP_TRY(dgemm_i8(st, dp_LinvT, dp_K, Kc, ldn, DG_TRI_UPPER, 0, n, false, 0));
    } else if (nc > 0) {
        GP_TRY(gemm_f64(st, false, false, G(n, nc, n, Linv, ldn, Kc, ldn, K2c, ldn, 1.0, 0.0, TRI_A_LOWER)));   // :19
        GP_TRY(launch_fstar_sd(st, K2c, ldn, n, nc, s + c0));                                                   // :20
        GP_TRY(gemm_f64(st, true, false, G(n, nc, n, Linv, ldn, K2c, ldn, Kc, ldn, 1.0, 0.0, TRI_A_UPPER)));
    }
    GP_TRY(gather_solves(st));
    toc_on(b, st);
    return GPIRT_B200_OK;
}

// f_star = draw_fstar(f, theta, theta_star, cholS, mu_star)                         gpirtMCMC.cpp:69, draw-fstar.cpp:10-31
int gpirt_b200_sampler::step_draw_fstar(uint32_t sweep, int accumulate) {
    const RngKey k = key_at(sweep);
    const int N = N_GRID;
    if (route != Route::LITERAL) {
        if (carry.solved == Carry::Solved::ALL) GP_CUDA(cudaStreamWaitEvent(stream, ev_solve, 0));   // done under the previous sweep's tail / this sweep's ESS
        else if (carry.solved == Carry::Solved::LOCAL) {   // this rank's slice was solved behind the factorisation: gather it now
            GP_CUDA(cudaStreamWaitEvent(stream, ev_solve, 0));
            tic(GPIRT_B200_T_TRSM);
            GP_TRY(gather_solves(stream));
            toc();
        } else GP_TRY(fstar_solves(stream));
        carry.solved = Carry::Solved::NONE;
        tic(GPIRT_B200_T_FSTAR_GEMM);
        if (use_i8gemm) {
            GP_TRY(dp_B.slice_kcontig(stream, f, ldn));
            GP_TRY(dgemm_i8(stream, dp_A, dp_B, fstar, ldN, DG_TRI_NONE, 0, n, false, FSTAR_GROUP_COLS));
        } else {
            GP_TRY(gemm_f64(stream, true, false, G(N, m, n, kstar, ldn, f, ldn, fstar, ldN, 1.0, 0.0, TRI_NONE)));
        }
        toc();
    } else {
        tic(GPIRT_B200_T_KSTAR);
        GP_TRY(launch_se_cov(stream, theta, n, theta_star, N, 0.0, false, kstar, ldn));          // :17
        toc();
        tic(GPIRT_B200_T_TRSM);
        GP_TRY(gemm_f64(stream, false, false, G(n, N, n, Linv, ldn, kstar, ldn, kstar2, ldn, 1.0, 0.0, TRI_A_LOWER)));   // :19
        GP_TRY(launch_fstar_sd(stream, kstar2, ldn, n, N, s));                                   // :20
        // literal: alpha_j = L^-T (L^-1 f_j) for every item (:3-8,:24), mean_j = K*^T alpha_j (:25)
        GP_TRY(gemm_f64(stream, false, false, G(n, m, n, Linv, ldn, f, ldn, Z, ldn, 1.0, 0.0, TRI_A_LOWER)));
        GP_TRY(gemm_f64(stream, true, false, G(n, m, n, Linv, ldn, Z, ldn, nu, ldn, 1.0, 0.0, TRI_A_UPPER)));
        toc();
        tic(GPIRT_B200_T_FSTAR_GEMM);
        GP_TRY(gemm_f64(stream, true, false, G(N, m, n, kstar, ldn, nu, ldn, fstar, ldN, 1.0, 0.0, TRI_NONE)));
        toc();
    }
    tic(GPIRT_B200_T_FSTAR_DRAW);
    GP_CUDA(cudaMemcpyAsync(Dmat, fstar, (size_t)ldN * m * sizeof(double), cudaMemcpyDeviceToDevice, stream));  // keep means for tests
    GP_TRY(launch_fstar_finish(stream, fstar, ldN, N, m, s, beta, theta_star, k, item_offset, irf_sum, accumulate));  // :26-28
    toc();
    return GPIRT_B200_OK;
}

__global__ void k_sub_rowsum(double* logPt, int64_t ld, int N, int n, const double* rowsum) {
    const int k = blockIdx.y * blockDim.x + threadIdx.x, i = blockIdx.x;   // respondents on grid.x (n may exceed 65535)
    if (k < N && i < n) logPt[k + (int64_t)i * ld] -= rowsum[k];
}

// theta = draw_theta(theta_star, y, theta_prior, f_star, mu_star)                   gpirtMCMC.cpp:70, draw-theta.cpp:3-37
int gpirt_b200_sampler::step_draw_theta(uint32_t sweep) {
    const RngKey k = key_at(sweep);
    const int N = N_GRID;
    double* rowsum = logPt + (size_t)ldN * n;   // column n of the logP buffer (rides along in the all-reduce)
    tic(GPIRT_B200_T_THETA_PREP);
    GP_TRY(launch_theta_prep(stream, fstar, Dmat, ldN, N, m, partial, N_CHUNKS, rowsum));
    toc();
    tic(GPIRT_B200_T_THETA_GEMM);
    // logP^T[k,i] = 1/2 sum_j f*_kj y_ij   (y = 0 where missing)
    if (use_ti8) GP_TRY(ti8.run(stream, fstar, ldN, 0.5, logPt, ldN, false, false));
    else GP_TRY(gemm_f64(stream, false, true, G(N, n, m, fstar, ldN, yd, ldn, logPt, ldN, 0.5, 0.0, TRI_NONE)));
    const double* rs_for_draw = rowsum;
    if (has_missing) {  // - sum_j obs_ij D_kj with obs = |y|
        if (use_ti8) GP_TRY(ti8.run(stream, Dmat, ldN, -1.0, logPt, ldN, true, true));
        else GP_TRY(gemm_f64(stream, false, true, G(N, n, m, Dmat, ldN, yd, ldn, logPt, ldN, -1.0, 1.0, TRI_NONE, 1)));
        rs_for_draw = nullptr;
    }
    toc();
    if (comm.world > 1) {
        tic(GPIRT_B200_T_ALLREDUCE);
        if (!has_missing) {
            dim3 grid((unsigned)n, (unsigned)ceil_div(N, 256));
            GP_LAUNCH(k_sub_rowsum, grid, 256, 0, stream, logPt, ldN, N, n, rowsum);
        }
        rs_for_draw = nullptr;
        GP_TRY(comm_allreduce_sum_f64(comm, logPt, (size_t)ldN * n, stream));
        toc();
    }
    tic(GPIRT_B200_T_THETA_DRAW);
    GP_TRY(launch_theta_draw(stream, logPt, ldN, rs_for_draw, prior, theta_star, n, N, k, theta, theta_idx, status + 2));
    toc();
    return GPIRT_B200_OK;
}

// beta = draw_beta(beta, X, y, f, ...) with X.col(1) = the NEW theta                 gpirtMCMC.cpp:71-73, draw-beta.cpp
int gpirt_b200_sampler::step_draw_beta(uint32_t sweep) {
    tic(GPIRT_B200_T_BETA);
    GP_TRY(launch_beta(stream, beta, f, ldn, y8, ldy8, theta, pm, psd, pstep, n, m, key_at(sweep), item_offset, status + 1, work + 1, &beta_shape));
    toc();
    return GPIRT_B200_OK;
}

// initial draws, gpirtMCMC.cpp:18-41 (sweep counter 0): f_j = cholS z_j, beta ~ N(pm, psd), f* = draw_fstar(...)
int gpirt_b200_sampler::init_draws() {
    sweep_counter = 0;
    GP_TRY(step_draw_f(0));
    GP_TRY(launch_init_beta(stream, beta, pm, psd, m, key_at(0), item_offset));
    GP_TRY(step_draw_fstar(0, 0));
    return check_status();
}

// ESS with nu already in place (the product L z was accumulated behind the previous sweep's factorisation)
int gpirt_b200_sampler::ess_only(uint32_t sweep) {
    tic(GPIRT_B200_T_ESS);
    // beside the backward substitution: one CTA per item instead of the persistent CTAs (which own every SM until the item
    // queue is empty), so that the short kernels of the pass get SMs as item CTAs retire
    // and one notch below the pass in priority: an item CTA takes the whole register file of its SM, and at equal priority
    // the block scheduler drains the grid that was launched first — the pass would start when the ESS has ended
    int* queue = carry.ess_yields ? nullptr : work;
    LaunchPriority yield(carry.ess_yields ? prio_second : INT_MIN);
    carry.ess_yields = false;
    GP_TRY(launch_ess(stream, f, nu, ldn, y8, ldy8, theta, beta, n, m, key_at(sweep), item_offset, nprop, status + 1, queue, &ess_shape));
    toc();
    return GPIRT_B200_OK;
}

// End of sweep `sweep` with the next sweep's proposals prepared under the factorisation:
//   st_beta : Z(next) = Philox normals, then the beta step                                   (needs the new theta only)
//   stream  : K(theta,theta)+1e-3 I, right-looking Cholesky chain (+ its bulk stream), L^-1
//   st_lz   : after every lz_group finished block columns  nu[r0:, :] (+)= L[r0:, r0:r1] Z[r0:r1, :]
int gpirt_b200_sampler::rebuild_pipelined(uint32_t sweep, uint32_t next_sweep) {
    GP_CUDA(cudaEventRecord(ev_theta, stream));
    GP_CUDA(cudaStreamWaitEvent(st_beta, ev_theta, 0));
    {
        Seg sg = tic_on(GPIRT_B200_T_FILL_Z, st_beta);
        if (use_i8gemm)
            GP_TRY(launch_fill_normal_planes(st_beta, dp_B.planes, dp_B.scale, dp_B.rows_pad, dp_B.k_pad, n, m, key_at(next_sweep),
                                             P_ESS_Z, item_offset, nullptr, ldn));
        else GP_TRY(launch_fill_normal(st_beta, Z, n, m, ldn, key_at(next_sweep), P_ESS_Z, item_offset));
        toc_on(sg, st_beta);
        GP_CUDA(cudaEventRecord(ev_z, st_beta));
        Seg sb = tic_on(GPIRT_B200_T_BETA, st_beta);
        // one CTA per item here, not the persistent variant: its CTAs retire every few microseconds, so the chain's short
        // high-priority kernels get SMs (a persistent CTA owns the whole register file of its SM: measured +0.5 ms/sweep)
        GP_TRY(launch_beta(st_beta, beta, f, ldn, y8, ldy8, theta, pm, psd, pstep, n, m, key_at(sweep), item_offset, status + 1, nullptr, &beta_shape));
        toc_on(sb, st_beta);
        GP_CUDA(cudaEventRecord(ev_beta, st_beta));
    }
    tic(GPIRT_B200_T_KBUILD);
    GP_TRY(launch_se_cov(stream, theta, n, theta, n, 0.001, true, L, ldn));
    toc();
    const bool subst = route == Route::SUBST;
    if (subst) {   // K* for this rank's grid columns as soon as theta is known
        GP_CUDA(cudaStreamWaitEvent(st_trsm, ev_theta, 0));
        Seg a = tic_on(GPIRT_B200_T_KSTAR, st_trsm);
        GP_TRY(trsm_kstar(st_trsm));
        toc_on(a, st_trsm);
    }
    bool first = true;
    // Slices of the overlapped product.  Through L^-1 (one GPU): equal slices of lz_group = 16 panels — every slice pays
    // the fixed-point kernel's epilogue over all row tiles below it, and what is left after the last panel runs under the
    // inversion.  Substitution route (items sharded): nothing hides the remainder, so the slices shrink towards the end
    // (half of the panels, all but an eighth, the rest: ~1.5 % of the product is left behind the factorisation).  Eight
    // equal slices of 4 panels were measured and lost (4.6 -> 5.2 ms per sweep on 4 GPUs): the early panels' bulk updates
    // keep the whole GPU busy, and product slices that start there only delay the chain.
    // The schedule may depend on the route but never on the sharding itself: the slices are added in FP64, so their
    // boundaries are part of the rounding of nu, and a sharded run must reproduce the unsharded one bit for bit.
    const int nblk_all = (int)ceil_div(n, CHOL_NB);
    auto next_end = [&](int e) {
        if (!use_i8gemm || !subst) return min(nblk_all, e + lz_group);
        if (e < nblk_all / 2) return max(1, nblk_all / 2);
        const int tail_start = nblk_all - max(1, nblk_all / 8);
        return e < tail_start ? tail_start : nblk_all;
    };
    int lz_slice = 0, lz_prev_end = 0, lz_next_end = next_end(0);
    lookahead.after_panel = [&](int k, int nblk, cudaEvent_t done) -> int {
        if (subst) {   // forward substitution step k trails panel k
            GP_CUDA(cudaStreamWaitEvent(st_trsm, done, 0));
            Seg sg = tic_on(GPIRT_B200_T_TRSM, st_trsm);
            GP_TRY(trsm_fwd_step(st_trsm, k));
            if (k != nblk - 1) GP_TRY(invert_bwd_step(st_trsm, k));   // block inverses of the backward pass grow behind the panels
            toc_on(sg, st_trsm);
        }
        // a slice of the product ends after every lz_group panels.  (Shrinking the later slices geometrically so that less of
        // the product is left when the factorisation ends was measured and lost: every slice pays the fixed-point kernel's
        // epilogue over all row tiles below it, 9.4 -> 10.3 ms per sweep at C3.)
        if (k + 1 != lz_next_end && k != nblk - 1) return GPIRT_B200_OK;
        const int g = lz_slice++;
        const int r0 = lz_prev_end * CHOL_NB, r1 = min(n, (k + 1) * CHOL_NB);
        lz_prev_end = k + 1;
        lz_next_end = next_end(lz_prev_end);
        if (first) {
            GP_CUDA(cudaStreamWaitEvent(st_lz, ev_z, 0));
            first = false;
        }
        GP_CUDA(cudaStreamWaitEvent(st_lz, done, 0));
        Seg sg = tic_on(GPIRT_B200_T_LZ_GEMM, st_lz);
        if (use_i8gemm) {
            GP_TRY(dp_L.slice_mcontig(st_lz, L, ldn, true, r0, r1, L_FIXED_EXP));
            GP_TRY(dgemm_i8(st_lz, dp_L, dp_B, nu, ldn, DG_TRI_LOWER, r0, r1, g != 0, LZ_GROUP_COLS, false));
        } else {
            GemmArgs a;
            a.M = n - r0; a.N = m; a.K = r1 - r0;
            a.A = L + r0 + (int64_t)r0 * ldn; a.lda = ldn; a.B = Z + r0; a.ldb = ldn; a.C = nu + r0; a.ldc = ldn;
            a.alpha = 1.0; a.beta = (g == 0) ? 0.0 : 1.0; a.tri = TRI_A_LOWER;
            GP_TRY(gemm_f64(st_lz, false, false, a));
        }
        toc_on(sg, st_lz);
        if (k == nblk - 1) GP_CUDA(cudaEventRecord(ev_lz, st_lz));
        return GPIRT_B200_OK;
    };
    tic(GPIRT_B200_T_CHOL);
    int rc = potrf_lower_rl(stream, L, ldn, n, Dinv, ldn, status, chol_flags, &lookahead);
    lookahead.after_panel = nullptr;
    GP_TRY(rc);
    toc();
    if (!subst) {
        tic(GPIRT_B200_T_TRTRI);
        GP_TRY(trtri_lower(stream, L, ldn, n, Dinv, ldn, Linv, ldn, Tmp, ldn));
        toc();
    } else {   // the forward steps join here; the backward substitution starts with the next sweep, beside its ESS
        GP_CUDA(cudaEventRecord(ev_fwd, st_trsm));
        GP_CUDA(cudaStreamWaitEvent(stream, ev_fwd, 0));
    }
    GP_CUDA(cudaStreamWaitEvent(stream, ev_lz, 0));
    GP_CUDA(cudaStreamWaitEvent(stream, ev_beta, 0));
    carry.nu_ready = true;
    carry.nu_sweep = next_sweep;
    // sharded, the solves through L^-1 run in the next sweep's draw_fstar: all ranks gather their slices there
    carry.start = subst ? Carry::Start::BWD
                : (route == Route::LINV && comm.world <= 1) ? Carry::Start::LINV_SOLVES : Carry::Start::NONE;
    return GPIRT_B200_OK;
}

int gpirt_b200_sampler::launch_deferred_solves() {
    const Carry::Start what = carry.start;
    carry.start = Carry::Start::NONE;
    if (what == Carry::Start::BWD) {
        // on the factorisation's bulk stream (idle now, same top priority as the ESS on the main stream: on the trailing
        // stream, one notch lower, the first kernel of the pass did not get an SM before the ESS had dispatched all of its
        // CTAs — 0.37 ms into the sweep on 4 GPUs)
        cudaStream_t st_tail = lookahead.aux ? lookahead.aux : st_trsm;
        GP_CUDA(cudaEventRecord(ev_linv, stream));
        GP_CUDA(cudaStreamWaitEvent(st_tail, ev_linv, 0));
        Seg sg = tic_on(GPIRT_B200_T_TRSM, st_tail);
        GP_TRY(trsm_bwd(st_tail, true));
        toc_on(sg, st_tail);
        GP_CUDA(cudaEventRecord(ev_solve, st_tail));
        carry.solved = Carry::Solved::LOCAL;
        carry.ess_yields = true;
    } else if (what == Carry::Start::LINV_SOLVES) {
        GP_CUDA(cudaEventRecord(ev_linv, stream));
        GP_CUDA(cudaStreamWaitEvent(st_lz, ev_linv, 0));
        GP_TRY(fstar_solves(st_lz));
        GP_CUDA(cudaEventRecord(ev_solve, st_lz));
        carry.solved = Carry::Solved::ALL;
    }
    return GPIRT_B200_OK;
}

__global__ void k_bump_sweep(uint32_t* sweep) { *sweep += 1u; }

int gpirt_b200_sampler::sweep_eager(uint32_t t, int accumulate) {
    const bool can_pipe = pipeline && ceil_div(n, CHOL_NB) > 2;   // the look-ahead factorisation needs > 2 panels
    GP_TRY(launch_deferred_solves());
    if (can_pipe && carry.nu_ready && carry.nu_sweep == t) GP_TRY(ess_only(t));
    else { carry.ess_yields = false; GP_TRY(step_draw_f(t)); }
    carry.nu_ready = false;
    GP_TRY(step_draw_fstar(t, accumulate));
    GP_TRY(step_draw_theta(t));
    if (can_pipe) return rebuild_pipelined(t, t + 1);
    GP_TRY(step_draw_beta(t));
    GP_TRY(step_rebuild());   // mu = X beta and mu* = X* beta (gpirtMCMC.cpp:74-75) are never materialised
    return GPIRT_B200_OK;
}

// A sweep as one CUDA graph launch: captured once per value of `accumulate` from the very launch sequence of sweep_eager
// (same kernels, same order, same draws: the sweep counter reaches the kernels through d_sweep, which the first node of
// the graph bumps).  At n = 100 a sweep is ~20 kernels of a few microseconds each; the graph removes the per-launch host
// cost and most of the gaps between dependent kernels.  The pipelined sweep is captured with its side streams: they fork
// from and join the capturing stream inside sweep_eager (launch_deferred_solves / rebuild_pipelined), every launch carries
// its stream's priority as a launch attribute (GP_LAUNCH) and the graph is instantiated with per-node priorities.
int gpirt_b200_sampler::sweep_graph(uint32_t t, int accumulate) {
    const int a = accumulate ? 1 : 0;
    if (!gexec[a]) {
        cudaGraph_t graph = nullptr;
        const int64_t counted = g_launch_count;   // recording a launch into a graph is not a launch
        capturing = true;
        capture_base = t;
        cudaError_t e = cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal);
        int rc = GPIRT_B200_OK;
        if (e == cudaSuccess) {
            GP_LAUNCH(k_bump_sweep, 1, 1, 0, stream, d_sweep);
            rc = sweep_eager(t, accumulate);
            e = cudaStreamEndCapture(stream, &graph);
            graph_carry[a] = carry;
            graph_carry[a].nu_sweep -= t;
        }
        capturing = false;
        g_launch_count = counted;
        if (rc == GPIRT_B200_OK && e == cudaSuccess) e = cudaGraphInstantiateWithFlags(&gexec[a], graph, cudaGraphInstantiateFlagUseNodePriority);   // per-node priorities = the priorities of the captured streams
        if (graph) cudaGraphDestroy(graph);
        if (rc != GPIRT_B200_OK || e != cudaSuccess) {   // not capturable on this driver: stay on the eager path for good
            cudaGetLastError();
            gexec[a] = nullptr;
            graph_enabled = false;
            return sweep_eager(t, accumulate);
        }
    }
    if (d_sweep_value != t - 1) {   // eager sweeps ran in between: resynchronise the device copy of the counter
        const uint32_t v = t - 1;
        GP_CUDA(cudaMemcpyAsync(d_sweep, &v, sizeof(v), cudaMemcpyHostToDevice, stream));
    }
    GP_CUDA(cudaGraphLaunch(gexec[a], stream));
    g_launch_count += graph_kernels;   // the kernels inside the graph still launch
    graph_replays += 1;
    d_sweep_value = t;
    carry = graph_carry[a];            // the host-side state the sweep leaves behind
    carry.nu_sweep += t;
    return GPIRT_B200_OK;
}

int gpirt_b200_sampler::sweep(int accumulate) {
    const uint32_t t = ++sweep_counter;
    const bool can_pipe = pipeline && ceil_div(n, CHOL_NB) > 2;
    // graph replay without per-step timers, after one eager sweep has done every lazy first-use initialisation (function
    // attributes, occupancy queries, the softplus table); the pipelined sweep only in its steady state (proposals and
    // solves prepared by the previous sweep), which is the state the captured launch sequence assumes
    const bool steady = !can_pipe || (carry.nu_ready && carry.nu_sweep == t && carry.start != Carry::Start::NONE);
    if (graph_enabled && !timing && warmed && route != Route::LITERAL && steady) return sweep_graph(t, accumulate);
    const int64_t before = g_launch_count;
    GP_TRY(sweep_eager(t, accumulate));
    graph_kernels = g_launch_count - before;
    warmed = true;
    return GPIRT_B200_OK;
}

void gpirt_b200_sampler::destroy() {
    if (stream) cudaStreamSynchronize(stream);
    for (auto& g : gexec) if (g) { cudaGraphExecDestroy(g); g = nullptr; }
    flush_timers();
    for (auto e : pool) cudaEventDestroy(e);
    pool.clear();
    for (auto e : lookahead.ev_panel) cudaEventDestroy(e);
    for (auto e : lookahead.ev_bulk) cudaEventDestroy(e);
    lookahead.ev_panel.clear(); lookahead.ev_bulk.clear();
    if (lookahead.aux) { cudaStreamSynchronize(lookahead.aux); cudaStreamDestroy(lookahead.aux); lookahead.aux = nullptr; }
    for (cudaStream_t* q : {&st_beta, &st_lz, &st_trsm}) if (*q) { cudaStreamSynchronize(*q); cudaStreamDestroy(*q); *q = nullptr; }
    for (cudaEvent_t* e : {&ev_theta, &ev_z, &ev_beta, &ev_lz, &ev_linv, &ev_solve, &ev_fwd}) if (*e) { cudaEventDestroy(*e); *e = nullptr; }
    dump_stamps();
    if (d_stamps) { cudaFree(d_stamps); d_stamps = nullptr; }
    if (trace_file) { fclose(trace_file); trace_file = nullptr; }
    if (trace_ref) { cudaEventDestroy(trace_ref); trace_ref = nullptr; }
    comm_destroy(comm);
    ti8.destroy();
    dp_L.destroy(); dp_A.destroy(); dp_B.destroy(); dp_Linv.destroy(); dp_LinvT.destroy(); dp_K.destroy();
    void* ptrs[] = {d_sweep, work, y8, yd, theta, theta_star, prior, beta, pm, psd, pstep, L, Dinv, f, Z, nu, fstar, Dmat, irf_sum,
                    kstar, s, logPt, partial, nprop, theta_idx, status, counters, Linv, Tmp, kstar2, chol_flags, splitk_ws, splitk_count};
    for (void* p : ptrs) pool_free(p, stream);
    if (stream) cudaStreamSynchronize(stream);
    if (stream) cudaStreamDestroy(stream);
    stream = nullptr;
}

// ----------------------------------------------------------------------------------------------------------------------
// Host side of draw storage: the caller's f array is ordinary pageable (R-allocated) memory, never touched before.
// A slice goes device -> pinned bounce buffer in chunks over PCIe by DMA, and a few host threads copy each chunk into
// the caller's array as soon as its DMA has landed (first-touch page faults are spread over the threads).
// ----------------------------------------------------------------------------------------------------------------------
namespace {
struct Bounce {
    double* buf[2] = {nullptr, nullptr};
    size_t cap = 0;
    std::vector<cudaEvent_t> ev[2];   // one event per DMA piece, per buffer
    // small pinned staging of a call (theta | beta of a slot, twice; status words + agreement ring): kept across calls like
    // the bounce buffers, so that a call neither pins nor unpins host memory (cudaFreeHost synchronises the device)
    double* small[2] = {nullptr, nullptr};
    size_t small_cap = 0;
    int* poll = nullptr;
    static constexpr size_t POLL_BYTES = 8 * sizeof(int) + 8 * sizeof(double);
    int ensure_small(size_t count) {
        if (!poll && cudaHostAlloc((void**)&poll, POLL_BYTES, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); poll = nullptr; return GPIRT_B200_ERR_NOMEM; }
        if (count <= small_cap) return GPIRT_B200_OK;
        for (auto& p : small) { if (p) cudaFreeHost(p); p = nullptr; }
        small_cap = 0;
        for (auto& p : small)
            if (cudaHostAlloc((void**)&p, count * sizeof(double), cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return GPIRT_B200_ERR_NOMEM; }
        small_cap = count;
        return GPIRT_B200_OK;
    }
    void release() {
        for (auto& p : buf) { if (p) cudaFreeHost(p); p = nullptr; }
        for (auto& p : small) { if (p) cudaFreeHost(p); p = nullptr; }
        if (poll) { cudaFreeHost(poll); poll = nullptr; }
        cap = small_cap = 0;
    }
    ~Bounce() { for (auto p : buf) if (p) cudaFreeHost(p); }
    int ensure(size_t count) {
        if (count <= cap) return GPIRT_B200_OK;
        for (auto& p : buf) { if (p) cudaFreeHost(p); p = nullptr; }
        cap = 0;
        for (auto& p : buf)
            if (cudaHostAlloc((void**)&p, count * sizeof(double), cudaHostAllocDefault) != cudaSuccess) {
                cudaGetLastError();
                return GPIRT_B200_ERR_NOMEM;
            }
        cap = count;
        return GPIRT_B200_OK;
    }
};
Bounce g_bounce;        // process-wide, reused across calls (2 x n*m*8 bytes of pinned memory once f draws are stored)
std::mutex g_bounce_mu; // held by a gpirt_b200_mcmc call for its whole duration (concurrent calls in one process take turns)

// host copy threads of one storage worker: one process per GPU on the same host, and the chains of one call, share the cores
int host_threads_for_copy(int chains) {
    const char* e = getenv("GPIRT_COPY_THREADS");
    int t = e ? atoi(e) : (int)std::min(12u, std::max(1u, std::thread::hardware_concurrency() * 3 / 4));
    const char* ws = getenv("WORLD_SIZE");
    const int share = (ws ? std::max(1, atoi(ws)) : 1) * chains;
    if (!e && share > 1) t = std::max(2, t / share);
    return t < 1 ? 1 : (t > 32 ? 32 : t);
}

// dst (pageable host) <- src (device), count doubles, via bounce buffer `b` on `stream`, in two phases so that the DMA of
// the NEXT slice (other buffer) can be enqueued before the copy threads start on this one:
//   bounce_issue   enqueues the DMA pieces and one event per piece
//   bounce_finish  copy threads pick the pieces up as they land
// Pieces are 4 MiB and start on 2 MiB boundaries of the DESTINATION: a slice lands in ~80 pieces, so the copy of the last
// piece — the only part that cannot overlap the DMA — is 4 MiB by one thread (with 32 MiB pieces one thread spent 8-20 ms
// on the last one after the DMA had finished: first-touch copies run at 1.5 GB/s per thread on 4 KiB pages, ~4 GB/s on
// huge pages; tools/host_store_probe.cpp), and a huge page of the destination is first touched by exactly one thread.
// `bo` is g_bounce (its caller holds g_bounce_mu) or bounce buffers a call owns; `threads` host threads copy.
struct BounceXfer {
    std::vector<size_t> cut;   // piece boundaries in doubles
    double* dst = nullptr;
    bool staged = false;       // false: no pinned memory, the copy was done by the driver in bounce_issue
    Bounce* bo = nullptr;
    int threads = 1;
};
int bounce_issue(Bounce& bo, int threads, double* dst, const double* src, size_t count, int b, cudaStream_t stream, BounceXfer& x) {
    x.dst = dst; x.cut.clear(); x.staged = false; x.bo = &bo; x.threads = threads;
    if (bo.ensure(count) != GPIRT_B200_OK) {   // no pinned memory: plain (driver-staged) copy
        GP_CUDA(cudaMemcpyAsync(dst, src, count * sizeof(double), cudaMemcpyDeviceToHost, stream));
        GP_CUDA(cudaStreamSynchronize(stream));
        return GPIRT_B200_OK;
    }
    const size_t piece = (size_t)4 << 20, huge = (size_t)2 << 20;   // bytes
    const uintptr_t d0 = (uintptr_t)dst, d1 = d0 + count * sizeof(double);
    x.cut.push_back(0);
    uintptr_t next = ((d0 + huge) & ~(uintptr_t)(huge - 1));        // first 2 MiB boundary after the start
    if (next - d0 < huge / 2) next += piece - huge;                   // no tiny first piece
    while (next < d1) { x.cut.push_back((next - d0) / sizeof(double)); next += piece; }
    x.cut.push_back(count);
    const int npieces = (int)x.cut.size() - 1;
    while ((int)bo.ev[b].size() < npieces) {
        cudaEvent_t e;
        GP_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        bo.ev[b].push_back(e);
    }
    double* bb = bo.buf[b];
    for (int c = 0; c < npieces; ++c) {
        GP_CUDA(cudaMemcpyAsync(bb + x.cut[c], src + x.cut[c], (x.cut[c + 1] - x.cut[c]) * sizeof(double), cudaMemcpyDeviceToHost, stream));
        GP_CUDA(cudaEventRecord(bo.ev[b][c], stream));
    }
    x.staged = true;
    return GPIRT_B200_OK;
}
int bounce_finish(int b, BounceXfer& x) {
    if (!x.staged) return GPIRT_B200_OK;
    const int npieces = (int)x.cut.size() - 1;
    const double* bb = x.bo->buf[b];
    const int T = std::min(x.threads, npieces);
    std::atomic<int> next{0};
    std::atomic<int> failed{0};
    auto work = [&]() {
        for (;;) {
            const int c = next.fetch_add(1);
            if (c >= npieces) break;
            if (cudaEventSynchronize(x.bo->ev[b][c]) != cudaSuccess) { failed = 1; break; }
            std::memcpy(x.dst + x.cut[c], bb + x.cut[c], (x.cut[c + 1] - x.cut[c]) * sizeof(double));
        }
    };
    std::vector<std::thread> th;
    for (int t = 1; t < T; ++t) th.emplace_back(work);
    work();
    for (auto& t : th) t.join();
    x.staged = false;
    if (failed) { set_last_error("device-to-host copy of a draw slice failed"); return GPIRT_B200_ERR_CUDA; }
    return GPIRT_B200_OK;
}
int chunked_d2h(Bounce& bo, int threads, double* dst, const double* src, size_t count, int b, cudaStream_t stream) {
    BounceXfer x;
    GP_TRY(bounce_issue(bo, threads, dst, src, count, b, stream, x));
    return bounce_finish(b, x);
}
}  // namespace

// ======================================================================================================================
// C ABI
// ======================================================================================================================
extern "C" {

const char* gpirt_b200_strerror(int status) {
    switch (status) {
        case GPIRT_B200_OK: return "ok";
        case GPIRT_B200_ERR_ARG: return "invalid argument";
        case GPIRT_B200_ERR_CUDA: return "CUDA error (no device or runtime failure)";
        case GPIRT_B200_ERR_NOT_PD: return "chol(): decomposition failed";
        case GPIRT_B200_ERR_INTERRUPT: return "interrupted";
        case GPIRT_B200_ERR_Y_VALUE: return "response matrix holds values other than 1, -1, NA";
        case GPIRT_B200_ERR_ESS: return "elliptical slice sampler did not terminate";
        case GPIRT_B200_ERR_NCCL: return "NCCL error";
        case GPIRT_B200_ERR_NOMEM: return "out of device memory";
        default: return "unknown status";
    }
}
const char* gpirt_b200_last_error(void) { return gpirt::last_error(); }

int gpirt_b200_release_memory(void) {
    GP_TRY(comm_shutdown());
    {
        std::lock_guard<std::mutex> lock(g_bounce_mu);
        g_bounce.release();
    }
    int dev = 0;
    GP_CUDA(cudaGetDevice(&dev));
    cudaMemPool_t pool;
    GP_CUDA(cudaDeviceGetDefaultMemPool(&pool, dev));
    GP_CUDA(cudaDeviceSynchronize());
    GP_CUDA(cudaMemPoolTrimTo(pool, 0));
    return GPIRT_B200_OK;
}

int gpirt_b200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

int gpirt_b200_nccl_unique_id(void* out128) { return comm_unique_id(out128); }

int gpirt_b200_sampler_create(gpirt_b200_sampler** out, const double* y, int64_t n, int64_t m, const double* theta_init,
                              const double* pm, const double* psd, const double* pstep, const gpirt_b200_opts* opts) {
    if (!out) return GPIRT_B200_ERR_ARG;
    *out = nullptr;
    gpirt_b200_sampler* s = new gpirt_b200_sampler();
    int rc = s->create(y, n, m, theta_init, pm, psd, pstep, opts);
    if (rc != GPIRT_B200_OK) { s->destroy(); delete s; return rc; }
    *out = s;
    return GPIRT_B200_OK;
}

int gpirt_b200_sampler_init_draws(gpirt_b200_sampler* s) { return s ? s->init_draws() : GPIRT_B200_ERR_ARG; }

int gpirt_b200_sampler_sweep(gpirt_b200_sampler* s, int n_sweeps, int accumulate_irf, float* elapsed_ms) {
    if (!s || n_sweeps < 0) return GPIRT_B200_ERR_ARG;
    struct Events {
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        ~Events() { if (e0) cudaEventDestroy(e0); if (e1) cudaEventDestroy(e1); }
    } ev;
    GP_CUDA(cudaEventCreate(&ev.e0)); GP_CUDA(cudaEventCreate(&ev.e1));
    GP_CUDA(cudaEventRecord(ev.e0, s->stream));
    for (int t = 0; t < n_sweeps; ++t) GP_TRY(s->sweep(accumulate_irf));
    GP_CUDA(cudaEventRecord(ev.e1, s->stream));
    cudaError_t e = cudaStreamSynchronize(s->stream);
    if (e != cudaSuccess) { set_last_error("sweep failed: %s", cudaGetErrorString(e)); return GPIRT_B200_ERR_CUDA; }
    if (elapsed_ms) cudaEventElapsedTime(elapsed_ms, ev.e0, ev.e1);
    return s->check_status();
}

int gpirt_b200_sampler_step(gpirt_b200_sampler* s, int step, uint32_t sweep) {
    if (!s) return GPIRT_B200_ERR_ARG;
    s->drop_carry();
    int rc;
    switch (step) {
        case GPIRT_B200_STEP_DRAW_F: rc = s->step_draw_f(sweep); break;
        case GPIRT_B200_STEP_DRAW_FSTAR: rc = s->step_draw_fstar(sweep, 0); break;
        case GPIRT_B200_STEP_DRAW_THETA: rc = s->step_draw_theta(sweep); break;
        case GPIRT_B200_STEP_DRAW_BETA: rc = s->step_draw_beta(sweep); break;
        case GPIRT_B200_STEP_REBUILD: rc = s->step_rebuild(); break;
        default: return GPIRT_B200_ERR_ARG;
    }
    if (rc != GPIRT_B200_OK) return rc;
    return s->check_status();
}

static int field_shape(gpirt_b200_sampler* s, int field, double** dev, int64_t* ld, int* rows, int* cols) {
    const int N = N_GRID;
    switch (field) {
        case GPIRT_B200_THETA: *dev = s->theta; *ld = s->ldn; *rows = s->n; *cols = 1; return 0;
        case GPIRT_B200_BETA: *dev = s->beta; *ld = 2; *rows = 2; *cols = s->m; return 0;
        case GPIRT_B200_F: *dev = s->f; *ld = s->ldn; *rows = s->n; *cols = s->m; return 0;
        case GPIRT_B200_FSTAR: *dev = s->fstar; *ld = s->ldN; *rows = N; *cols = s->m; return 0;
        case GPIRT_B200_CHOL: *dev = s->L; *ld = s->ldn; *rows = s->n; *cols = s->n; return 0;
        case GPIRT_B200_NU: *dev = s->nu; *ld = s->ldn; *rows = s->n; *cols = s->m; return 0;
        case GPIRT_B200_FSTAR_S: *dev = s->s; *ld = s->ldN; *rows = N; *cols = 1; return 0;
        case GPIRT_B200_FSTAR_MEAN: *dev = s->Dmat; *ld = s->ldN; *rows = N; *cols = s->m; return 0;
        case GPIRT_B200_IRF_SUM: *dev = s->irf_sum; *ld = s->ldN; *rows = N; *cols = s->m; return 0;
        default: return -1;
    }
}

int gpirt_b200_sampler_get(gpirt_b200_sampler* s, int field, double* host_out) {
    if (!s || !host_out) return GPIRT_B200_ERR_ARG;
    const int N = N_GRID;
    if (field == GPIRT_B200_LOGP) {  // n x N, log-likelihood part only (host transposes the device's N x n layout)
        std::vector<double> t((size_t)N * (s->n + 1));
        GP_TRY(download_padded(t.data(), s->logPt, s->ldN, N, s->n + 1, s->stream));
        GP_CUDA(cudaStreamSynchronize(s->stream));
        const bool sub = !s->has_missing && s->comm.world <= 1;
        for (int i = 0; i < s->n; ++i)
            for (int k = 0; k < N; ++k)
                host_out[(size_t)k * s->n + i] = t[(size_t)i * N + k] - (sub ? t[(size_t)s->n * N + k] : 0.0);
        return GPIRT_B200_OK;
    }
    if (field == GPIRT_B200_THETA_IDX || field == GPIRT_B200_ESS_NPROP) {
        const int cnt = field == GPIRT_B200_THETA_IDX ? s->n : s->m;
        std::vector<int> t(cnt);
        GP_CUDA(cudaMemcpyAsync(t.data(), field == GPIRT_B200_THETA_IDX ? s->theta_idx : s->nprop, cnt * sizeof(int),
                                cudaMemcpyDeviceToHost, s->stream));
        GP_CUDA(cudaStreamSynchronize(s->stream));
        for (int i = 0; i < cnt; ++i) host_out[i] = (double)t[i];
        return GPIRT_B200_OK;
    }
    double* dev; int64_t ld; int rows, cols;
    if (field_shape(s, field, &dev, &ld, &rows, &cols)) return GPIRT_B200_ERR_ARG;
    GP_TRY(download_padded(host_out, dev, ld, rows, cols, s->stream));
    GP_CUDA(cudaStreamSynchronize(s->stream));
    return GPIRT_B200_OK;
}

int gpirt_b200_sampler_set(gpirt_b200_sampler* s, int field, const double* host_in) {
    if (!s || !host_in) return GPIRT_B200_ERR_ARG;
    double* dev; int64_t ld; int rows, cols;
    if (field_shape(s, field, &dev, &ld, &rows, &cols)) return GPIRT_B200_ERR_ARG;
    s->drop_carry();
    GP_TRY(upload_padded(dev, ld, host_in, rows, cols, s->stream));
    GP_CUDA(cudaStreamSynchronize(s->stream));
    return GPIRT_B200_OK;
}

int gpirt_b200_sampler_timings(gpirt_b200_sampler* s, double* ms, int64_t* calls, int reset) {
    if (!s) return GPIRT_B200_ERR_ARG;
    for (int i = 0; i < GPIRT_B200_TIMER_COUNT; ++i) {
        if (ms) ms[i] = s->ms[i];
        if (calls) calls[i] = s->calls[i];
        if (reset) { s->ms[i] = 0.0; s->calls[i] = 0; }
    }
    return GPIRT_B200_OK;
}

int gpirt_b200_sampler_set_timing(gpirt_b200_sampler* s, int enabled) {
    if (!s) return GPIRT_B200_ERR_ARG;
    s->timing = enabled != 0;
    return GPIRT_B200_OK;
}

int gpirt_b200_sampler_set_pipeline(gpirt_b200_sampler* s, int enabled) {
    if (!s) return GPIRT_B200_ERR_ARG;
    s->pipeline = enabled != 0;
    s->drop_graphs();
    s->drop_carry();
    return GPIRT_B200_OK;
}

// Time of K(theta, theta) + 0.001 I and its factorisation alone (no other work on the GPU), per repetition, either as the
// eager launch sequence or replayed as a CUDA graph of the same sequence (the way a sweep runs it inside gpirt_b200_mcmc).
// Measurement facility for bench.py; the factor is left in place (same theta: same L).
int gpirt_b200_sampler_time_factorisation(gpirt_b200_sampler* s, int reps, int as_graph, float* ms_per_rep) {
    if (!s || reps <= 0 || !ms_per_rep) return GPIRT_B200_ERR_ARG;
    GP_TRY(s->check_status());                              // drains every stream of the sampler
    s->drop_carry();
    const bool timing_was = s->timing;
    s->timing = false;
    struct Restore { gpirt_b200_sampler* s; bool t; ~Restore() { s->timing = t; } } restore{s, timing_was};
    auto once = [&]() -> int {
        GP_TRY(launch_se_cov(s->stream, s->theta, s->n, s->theta, s->n, 0.001, true, s->L, s->ldn));
        return potrf_lower_rl(s->stream, s->L, s->ldn, s->n, s->Dinv, s->ldn, s->status, s->chol_flags, &s->lookahead);
    };
    GP_TRY(once());                                         // warm (lazy attribute set-up, events of the look-ahead)
    GP_CUDA(cudaStreamSynchronize(s->stream));
    cudaGraphExec_t exec = nullptr;
    if (as_graph) {
        cudaGraph_t graph = nullptr;
        const int64_t counted = g_launch_count;
        GP_CUDA(cudaStreamBeginCapture(s->stream, cudaStreamCaptureModeThreadLocal));
        const int rc = once();
        const cudaError_t e = cudaStreamEndCapture(s->stream, &graph);
        g_launch_count = counted;
        if (rc != GPIRT_B200_OK || e != cudaSuccess) { if (graph) cudaGraphDestroy(graph); cudaGetLastError(); set_last_error("the factorisation could not be captured"); return GPIRT_B200_ERR_CUDA; }
        const cudaError_t ei = cudaGraphInstantiateWithFlags(&exec, graph, cudaGraphInstantiateFlagUseNodePriority);
        cudaGraphDestroy(graph);
        if (ei != cudaSuccess) { cudaGetLastError(); set_last_error("the factorisation graph could not be instantiated"); return GPIRT_B200_ERR_CUDA; }
        GP_CUDA(cudaGraphLaunch(exec, s->stream));          // one untimed replay
        GP_CUDA(cudaStreamSynchronize(s->stream));
    }
    cudaEvent_t e0, e1;
    GP_CUDA(cudaEventCreate(&e0)); GP_CUDA(cudaEventCreate(&e1));
    int rc = GPIRT_B200_OK;
    cudaEventRecord(e0, s->stream);
    for (int r = 0; r < reps && rc == GPIRT_B200_OK; ++r) {
        if (exec) { if (cudaGraphLaunch(exec, s->stream) != cudaSuccess) rc = GPIRT_B200_ERR_CUDA; }
        else rc = once();
    }
    cudaEventRecord(e1, s->stream);
    const cudaError_t es = cudaStreamSynchronize(s->stream);
    float t = 0.f;
    if (es == cudaSuccess) cudaEventElapsedTime(&t, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (exec) cudaGraphExecDestroy(exec);
    if (rc != GPIRT_B200_OK || es != cudaSuccess) { cudaGetLastError(); set_last_error("timing the factorisation failed"); return GPIRT_B200_ERR_CUDA; }
    *ms_per_rep = t / reps;
    return s->check_status();
}

int64_t gpirt_b200_sampler_launches(gpirt_b200_sampler* s) { return s ? g_launch_count - s->launches_at_create : 0; }
int gpirt_b200_sampler_uses(gpirt_b200_sampler* s, int feature) {
    if (!s) return -1;
    if (feature == 0) return s->use_ti8 ? 1 : 0;
    if (feature == 1) return s->use_i8gemm ? 1 : 0;
    if (feature == 2) return s->ess_shape;
    if (feature == 3) return s->beta_shape;
    if (feature == 4) return s->route == gpirt_b200_sampler::Route::SUBST ? 1 : 0;
    if (feature == 5) return (int)std::min<int64_t>(s->graph_replays, INT_MAX);
    return -1;
}

void gpirt_b200_sampler_destroy(gpirt_b200_sampler* s) {
    if (!s) return;
    s->destroy();
    delete s;
}

// ----------------------------------------------------------------------------------------------------------------------
// gpirtMCMC(): src/gpirtMCMC.cpp:5-117
// ----------------------------------------------------------------------------------------------------------------------
// Draw storage runs on its own host thread: the caller's arrays are fresh pageable memory, and a slice of f draws
// (n m doubles) takes 2-3 sweeps' worth of time to land there.  The sampling thread only snapshots the state on the device
// (two buffers) and hands the slot to this worker, which waits for the snapshot, moves it over PCIe and into the caller's
// arrays while the sampling thread keeps the GPU's launch queue full.  With thinned draws the stores disappear behind
// the sweeps; with every draw stored the worker is the bottleneck and the sampling thread waits for a free buffer.
namespace {
struct StoreWorker {
    std::mutex mu;
    std::condition_variable cv;
    std::deque<int> jobs;              // slots to drain, in order
    int drained[2] = {-1, -1};         // last slot drained from snapshot buffer b (a buffer is free when nothing is queued on it)
    int queued[2] = {-1, -1};          // last slot queued on buffer b
    bool quit = false;
    int rc = GPIRT_B200_OK;            // first failure of a drain
    std::string error;
    std::function<int(int)> issue;     // enqueue the device-to-host transfers of a slot        (both run on the worker thread)
    std::function<int(int)> finish;    // land them in the caller's arrays
    int issued = -1;                   // last slot whose transfers are enqueued
    std::thread th;
    int device = 0;
    double busy_s = 0.0;

    void start() {
        th = std::thread([this] {
            cudaSetDevice(device);
            for (;;) {
                int slot;
                {
                    std::unique_lock<std::mutex> lk(mu);
                    cv.wait(lk, [this] { return quit || !jobs.empty(); });
                    if (jobs.empty()) return;          // quit with nothing left
                    slot = jobs.front();
                    jobs.pop_front();
                }
                int r = GPIRT_B200_OK;
                {
                    std::lock_guard<std::mutex> lk(mu);
                    r = rc;
                }
                if (r == GPIRT_B200_OK) {              // after a failure the remaining jobs are dropped
                    if (issued != slot) { r = issue(slot); issued = slot; }
                    if (r == GPIRT_B200_OK) {          // the next slot's DMA (other buffers) runs under this slot's host copies
                        int nxt = -1;
                        {
                            std::lock_guard<std::mutex> lk(mu);
                            if (!jobs.empty()) nxt = jobs.front();
                        }
                        if (nxt >= 0 && (nxt & 1) != (slot & 1)) { r = issue(nxt); issued = nxt; }
                    }
                    if (r == GPIRT_B200_OK) r = finish(slot);
                    if (r != GPIRT_B200_OK) {
                        std::lock_guard<std::mutex> lk(mu);
                        rc = r;
                        error = last_error();
                    }
                }
                {
                    std::lock_guard<std::mutex> lk(mu);
                    drained[slot & 1] = slot;
                }
                cv.notify_all();
            }
        });
    }
    void push(int slot) {
        {
            std::lock_guard<std::mutex> lk(mu);
            jobs.push_back(slot);
            queued[slot & 1] = slot;
        }
        cv.notify_all();
    }
    void wait_buffer_free(int b) {       // the previous slot snapshotted into buffer b has reached the host
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return drained[b] == queued[b]; });
    }
    void wait_idle() { wait_buffer_free(0); wait_buffer_free(1); }
    int status(std::string* msg) {
        std::lock_guard<std::mutex> lk(mu);
        if (rc != GPIRT_B200_OK && msg) *msg = error;
        return rc;
    }
    void stop() {
        if (!th.joinable()) return;
        {
            std::lock_guard<std::mutex> lk(mu);
            quit = true;
            jobs.clear();
        }
        cv.notify_all();
        th.join();
    }
};
}  // namespace

static thread_local int64_t g_last_degenerate_theta = 0;
int64_t gpirt_b200_last_degenerate_theta(void) { return g_last_degenerate_theta; }

// running mean / sum of squared deviations of f over the sampling iterations (Welford), count = iterations so far incl. this
__global__ void __launch_bounds__(256) k_f_welford(const double* __restrict__ f, int64_t ld, int n, double count,
                                                   double* __restrict__ mean, double* __restrict__ m2) {
    const int i = blockIdx.y * blockDim.x + threadIdx.x, j = blockIdx.x;
    if (i >= n) return;
    const int64_t o = i + (int64_t)j * n;
    const double x = f[i + (int64_t)j * ld];
    const double mu = (count == 1.0) ? 0.0 : mean[o], q = (count == 1.0) ? 0.0 : m2[o];
    const double d = x - mu, mu2 = mu + d / count;
    mean[o] = mu2;
    m2[o] = fma(d, x - mu2, q);
}
__global__ void __launch_bounds__(256) k_f_sd(double* __restrict__ m2, size_t count_elems, double denom) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count_elems) m2[i] = sqrt(m2[i] / denom);   // denom = S - 1 (R's sd); S = 1 gives NaN like sd() of one value
}

namespace {
// Free device memory for a buffer of `need` bytes.  Memory the pool holds unused is free for this purpose: when short, the
// pool is handed back first.
int free_memory_for(double need, cudaStream_t st, size_t* free_b) {
    size_t total_b = 0;
    GP_CUDA(cudaMemGetInfo(free_b, &total_b));
    if (need > (double)*free_b) {
        int dev = 0;
        cudaMemPool_t pool;
        GP_CUDA(cudaStreamSynchronize(st));
        GP_CUDA(cudaGetDevice(&dev));
        GP_CUDA(cudaDeviceGetDefaultMemPool(&pool, dev));
        GP_CUDA(cudaMemPoolTrimTo(pool, 0));
        GP_CUDA(cudaMemGetInfo(free_b, &total_b));
    }
    return GPIRT_B200_OK;
}

// One chain of gpirtMCMC(): the sampler, its draw storage (snapshot buffers, copy stream, StoreWorker), the status polling
// and the on-device accumulators, driven by setup(), one iterate() per sweep and finish().  gpirt_b200_mcmc drives one;
// with opts.chains it drives several on one device, round-robin from the calling thread.  The progress callback belongs
// to the driver: a chain only learns of an interrupt through want_stop.
struct ChainRun {
    // arguments of the call (outputs already offset to this chain's block)
    const double* y; int64_t n, m; const double* theta_init; int S, B; const double *pm, *psd, *pstep;
    const gpirt_b200_opts* opts; double *theta_out, *beta_out, *f_out, *irf_out;
    Bounce* bo;                       // pinned staging: g_bounce, or a set the call owns
    int copy_threads;                 // host copy threads of the storage worker
    bool trace;                       // GPIRT_TIMING
    bool untraced = false;            // create() ignores GPIRT_TRACE (chains after the first)
    // several chains: this chain's trace of theta | beta (P x S, parameter-major) and its IRF half-chain states
    double* diag_trace = nullptr;
    double* diag_halves = nullptr;

    bool keep_f = true; int thin = 1;
    double *f_mean_out = nullptr, *f_sd_out = nullptr; bool summarise_f = false;
    gpirt_b200_fit* fit = nullptr; gpirt_b200_irf* irf = nullptr;
    int n_slots = 0; size_t nm = 0, n_small = 0; bool sharded = false;
    // resources, released by the destructor
    gpirt_b200_sampler* s = nullptr; cudaStream_t copy = nullptr; cudaEvent_t ev[2] = {nullptr, nullptr};
    double* snap_f[2] = {nullptr, nullptr}; double* snap_small[2] = {nullptr, nullptr};
    double *f_mean = nullptr, *f_m2 = nullptr, *agree_dev = nullptr; int* h_poll = nullptr; StoreWorker* worker = nullptr;
    double* h_small[2] = {nullptr, nullptr}; cudaEvent_t ev_small[2] = {nullptr, nullptr};
    double* pred_acc = nullptr; int8_t* pred_code = nullptr; double* pred_aux = nullptr;   // opts.fit
    double* irf_buf = nullptr; double* snap_fs[2] = {nullptr, nullptr};                     // opts.irf
    gpirt_b200_ppc* ppc = nullptr; PpcChi2 ppc_chi2; PpcPairs ppc_pairs;                     // opts.ppc
    // state of the run
    double* h_ring = nullptr; volatile int* w_poll = nullptr; int agree_count = 0;
    static constexpr int PRED_CHUNKS = 64;
    size_t pred_plane = 0;
    double *pred_stats = nullptr, *pred_partial = nullptr, *pred_resp = nullptr;
    int64_t irf_cells = 0; size_t irf_plane = 0; double* fs_out = nullptr; bool irf_bands = false; IrfBandPlan irf_plan{};
    double *irf_lo = nullptr, *irf_hi = nullptr;
    BounceXfer xfer[2];
    bool want_stop = false; int stop_code = GPIRT_B200_OK; int n_summarised = 0;
    int64_t degenerate = 0;           // theta draws with a degenerate grid CDF (finish)
    double t_a = 0.0, t_b = 0.0, t_c = 0.0, t_d = 0.0;

    static double now() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec + 1e-9 * ts.tv_nsec; }

    ~ChainRun() {
        const double t0 = now();
        if (worker) {   // before anything it uses goes away
            worker->stop();
            if (trace) fprintf(stderr, "gpirt_b200_mcmc: storage thread joined in %.3fs\n", now() - t0);
            delete worker;
        }
        if (!s) return;
        if (copy) { cudaStreamSynchronize(copy); cudaStreamDestroy(copy); }
        const double t1 = now();
        for (int i = 0; i < 2; ++i) if (ev_small[i]) cudaEventDestroy(ev_small[i]);   // h_small / h_poll belong to bo
        for (int i = 0; i < 2; ++i) { if (ev[i]) cudaEventDestroy(ev[i]); pool_free(snap_f[i], s->stream); pool_free(snap_small[i], s->stream); }
        pool_free(f_mean, s->stream); pool_free(f_m2, s->stream); pool_free(agree_dev, s->stream);
        pool_free(pred_acc, s->stream); pool_free(pred_code, s->stream); pool_free(pred_aux, s->stream);
        for (int i = 0; i < 2; ++i) pool_free(snap_fs[i], s->stream);
        if (irf_buf) { cudaStreamSynchronize(s->stream); cudaFree(irf_buf); }   // not the pool: GBs of tail buffers must not stay reserved after the call
        if (ppc_pairs.buf) { cudaStreamSynchronize(s->stream); ppc_pairs.destroy(); }   // likewise
        ppc_chi2.destroy();
        const double t2 = now();
        gpirt_b200_sampler_destroy(s);
        if (trace) fprintf(stderr, "gpirt_b200_mcmc: teardown worker/copy stream %.3fs, host + pool frees %.3fs, sampler %.3fs\n", t1 - t0, t2 - t1, now() - t2);
    }

    int d2h(double* dst, const double* src, size_t count, int b) { return chunked_d2h(*bo, copy_threads, dst, src, count, b, copy); }

    // snapshot(slot): main stream copies theta | beta (and f, tightly packed) into buffer slot & 1 and records the event
    int snapshot(int slot) {
        const int b = slot & 1;
        GP_CUDA(cudaMemcpyAsync(snap_small[b], s->theta, (size_t)n * sizeof(double), cudaMemcpyDeviceToDevice, s->stream));
        GP_CUDA(cudaMemcpyAsync(snap_small[b] + n, s->beta, 2 * (size_t)m * sizeof(double), cudaMemcpyDeviceToDevice, s->stream));
        if (keep_f)
            GP_CUDA(cudaMemcpy2DAsync(snap_f[b], (size_t)n * sizeof(double), s->f, s->ldn * sizeof(double), (size_t)n * sizeof(double),
                                      (size_t)m, cudaMemcpyDeviceToDevice, s->stream));
        if (fs_out)
            GP_CUDA(cudaMemcpy2DAsync(snap_fs[b], N_GRID * sizeof(double), s->fstar, s->ldN * sizeof(double), N_GRID * sizeof(double),
                                      (size_t)m, cudaMemcpyDeviceToDevice, s->stream));
        GP_CUDA(cudaEventRecord(ev[b], s->stream));
        return GPIRT_B200_OK;
    }

    // Stopping early (interrupt from the progress callback, failed Cholesky / ESS seen in the polled status words, a failed
    // store) must be a COMMON decision when items are sharded: a rank that returned alone would leave its peers blocked in
    // the next sweep's collectives.  Every rank therefore enqueues, every 8th iteration, a one-word all-reduce of its local
    // stop request on the sampler's stream and acts on the agreed value after the host sync that follows it — the same
    // program point on every rank.  An unsharded chain stops as soon as it sees a reason.
    int local_stop_code() {
        std::string msg;
        const int wrc = worker->status(&msg);
        if (wrc != GPIRT_B200_OK) { set_last_error("%s", msg.c_str()); return wrc; }
        if (h_poll[0] || w_poll[0]) { set_last_error("chol(): decomposition failed"); return GPIRT_B200_ERR_NOT_PD; }
        if (h_poll[1] || w_poll[1]) { set_last_error("elliptical slice sampler did not terminate (NaN log-likelihood?)"); return GPIRT_B200_ERR_ESS; }
        if (want_stop) { set_last_error("interrupted by the progress callback"); return GPIRT_B200_ERR_INTERRUPT; }
        return GPIRT_B200_OK;
    }
    int enqueue_agreement() {
        if (!sharded) return GPIRT_B200_OK;
        const double mine = local_stop_code() != GPIRT_B200_OK ? 1.0 : 0.0;   // pageable source: staged at call time
        GP_CUDA(cudaMemcpyAsync(agree_dev, &mine, sizeof(double), cudaMemcpyHostToDevice, s->stream));
        GP_TRY(comm_allreduce_sum_f64(s->comm, agree_dev, 1, s->stream));
        GP_CUDA(cudaMemcpyAsync(h_ring + (agree_count & 7), agree_dev, sizeof(double), cudaMemcpyDeviceToHost, s->stream));
        agree_count += 1;
        return GPIRT_B200_OK;
    }
    bool stop_now(int agreement) {   // after a host sync that covers agreement number `agreement`
        stop_code = local_stop_code();
        if (sharded) {
            if (agreement < 0 || h_ring[agreement & 7] == 0.0) return false;
            if (stop_code == GPIRT_B200_OK) { set_last_error("stopped: another rank was interrupted or failed"); stop_code = GPIRT_B200_ERR_INTERRUPT; }
            return true;
        }
        return stop_code != GPIRT_B200_OK;
    }
    // before each iteration: interrupt, failed store, failed chain seen by the worker (unsharded: sharded ranks agree later)
    bool stopped() { return !sharded && stop_now(-1); }

    int setup();
    int iterate(int iter);
    int finish();
};

int ChainRun::setup() {
    keep_f = !(opts && opts->skip_f_draws);
    thin = (opts && opts->thin > 1) ? opts->thin : 1;
    f_mean_out = opts ? opts->f_mean_out : nullptr;
    f_sd_out = opts ? opts->f_sd_out : nullptr;
    summarise_f = f_mean_out || f_sd_out;
    fit = opts ? opts->fit : nullptr;
    irf = opts ? opts->irf : nullptr;
    ppc = opts ? opts->ppc : nullptr;
    t_a = now();
    t_untraced_create = untraced;
    const int crc = gpirt_b200_sampler_create(&s, y, n, m, theta_init, pm, psd, pstep, opts);
    t_untraced_create = false;
    GP_TRY(crc);
    s->timing = false;
    t_b = now();
    // Draw storage overlaps the next sweep: after sweep t the state is snapshotted device-to-device (cheap), the host
    // enqueues sweep t+1, and only then blocks in the device-to-host copy of snapshot t on a second stream.
    n_slots = S / thin + 1;         // slot 0 = initial values, slot k = sampling iteration k * thin
    nm = (size_t)n * m;
    if (keep_f && !getenv("GPIRT_NO_HUGEPAGE_HINT")) {
        // the caller's f array is fresh pageable memory: ask for transparent huge pages on its interior so that the
        // first-touch faults of the draw stores are 2 MiB each instead of 4 KiB (advisory; ignored where THP is off).
        // On this pool's hosts 12 threads copy a 328 MB slice into fresh memory in 19 ms on 4 KiB pages and in 10 ms on
        // huge pages (tools/host_store_probe.cpp); numpy gives its large arrays the same hint, R's allocator does not.
        const uintptr_t a = ((uintptr_t)f_out + ((size_t)2 << 20) - 1) & ~(((uintptr_t)2 << 20) - 1);
        const uintptr_t b = ((uintptr_t)f_out + (size_t)n_slots * nm * sizeof(double)) & ~(((uintptr_t)2 << 20) - 1);
        if (b > a) madvise((void*)a, b - a, MADV_HUGEPAGE);
    }
    n_small = (size_t)n + 2 * (size_t)m;     // theta | beta of one slot
    GP_CUDA(cudaStreamCreateWithFlags(&copy, cudaStreamNonBlocking));
    if (bo->ensure_small(n_small) != GPIRT_B200_OK) { set_last_error("pinned host staging could not be allocated"); return GPIRT_B200_ERR_NOMEM; }
    for (int i = 0; i < 2; ++i) {
        h_small[i] = bo->small[i];
        GP_CUDA(cudaEventCreateWithFlags(&ev_small[i], cudaEventDisableTiming));
    }
    h_poll = bo->poll;
    std::memset(h_poll, 0, Bounce::POLL_BYTES);   // [0..3] status words polled by this thread, [4..7] by the
    h_ring = reinterpret_cast<double*>(h_poll + 8);      // storage worker, then a ring of 8 agreed stop flags
    w_poll = h_poll + 4;
    for (int i = 0; i < 2; ++i) {
        GP_CUDA(cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming));
        GP_TRY(pool_alloc((void**)&snap_small[i], n_small * sizeof(double), s->stream));
        if (keep_f) GP_TRY(pool_alloc((void**)&snap_f[i], nm * sizeof(double), s->stream));
    }
    if (summarise_f) {
        GP_TRY(pool_alloc((void**)&f_mean, nm * sizeof(double), s->stream));
        GP_TRY(pool_alloc((void**)&f_m2, nm * sizeof(double), s->stream));
    }
    sharded = s->comm.world > 1;
    if (sharded) GP_TRY(pool_alloc((void**)&agree_dev, sizeof(double), s->stream));
    // posterior predictive summaries: 3 accumulator planes (ldn x m), the cell code, per-item statistics, the per-respondent
    // partial sums, elpd per respondent + totals, and the illegal-value counter of y_holdout
    pred_plane = (size_t)s->ldn * m;
    if (fit) {
        GP_TRY(pool_alloc((void**)&pred_acc, 3 * pred_plane * sizeof(double), s->stream));
        GP_TRY(pool_alloc((void**)&pred_code, (size_t)s->ldy8 * m, s->stream));
        const size_t aux = (size_t)PRED_STATS * m + (size_t)PRED_CHUNKS * n + (size_t)n + PRED_STATS + 1;
        GP_TRY(pool_alloc((void**)&pred_aux, aux * sizeof(double), s->stream));
        pred_stats = pred_aux;
        pred_partial = pred_stats + (size_t)PRED_STATS * m;
        pred_resp = pred_partial + (size_t)PRED_CHUNKS * n;
        unsigned long long* n_bad = reinterpret_cast<unsigned long long*>(pred_resp + n + PRED_STATS);
        GP_CUDA(cudaMemsetAsync(n_bad, 0, sizeof(unsigned long long), s->stream));
        // y_holdout goes up through the first accumulator plane (not in use before the first sampling iteration)
        if (fit->y_holdout) GP_TRY(upload_pageable(pred_acc, fit->y_holdout, nm * sizeof(double), s->stream));
        GP_TRY(launch_predictive_code(s->stream, s->y8, s->ldy8, fit->y_holdout ? pred_acc : nullptr, (int)n, (int)m,
                                      pred_code, n_bad));
        unsigned long long bad = 0;
        GP_CUDA(cudaMemcpyAsync(&bad, n_bad, sizeof(bad), cudaMemcpyDeviceToHost, s->stream));
        GP_CUDA(cudaStreamSynchronize(s->stream));
        double bad_all = (double)bad;
        if (sharded) {   // every rank refuses together: one that returned alone would leave its peers in the first collective
            GP_CUDA(cudaMemcpyAsync(agree_dev, &bad_all, sizeof(double), cudaMemcpyHostToDevice, s->stream));
            GP_TRY(comm_allreduce_sum_f64(s->comm, agree_dev, 1, s->stream));
            GP_CUDA(cudaMemcpyAsync(&bad_all, agree_dev, sizeof(double), cudaMemcpyDeviceToHost, s->stream));
            GP_CUDA(cudaStreamSynchronize(s->stream));
        }
        if (bad_all != 0.0) {
            set_last_error("y_holdout holds %.0f values that are not +1, -1 or NA", bad_all);
            return GPIRT_B200_ERR_Y_VALUE;
        }
    }
    // IRF summaries: the Welford mean / M2 of P (2 planes of 1001 x m) and the tail heaps (K_lo + K_hi planes) in one
    // cudaMalloc, checked against the free device memory by arithmetic before the first sweep
    irf_cells = (int64_t)N_GRID * m;
    irf_plane = (size_t)irf_cells;
    fs_out = irf ? irf->fstar_draws : nullptr;
    irf_bands = irf && (irf->lower || irf->upper) && S > 0;
    irf_plan = irf_bands ? irf_band_plan(S, irf->band) : IrfBandPlan{};
    if (irf) {
        irf->band_bytes = 0;
        const double tail_bytes = 8.0 * (double)irf_cells * ((double)irf_plan.klo + (double)irf_plan.khi);
        const double need = tail_bytes + 16.0 * (double)irf_cells;
        size_t free_b = 0;
        GP_TRY(free_memory_for(need, s->stream, &free_b));
        double short_all = need > (double)free_b ? 1.0 : 0.0;
        if (sharded) {   // every rank refuses together, as for y_holdout
            GP_CUDA(cudaMemcpyAsync(agree_dev, &short_all, sizeof(double), cudaMemcpyHostToDevice, s->stream));
            GP_TRY(comm_allreduce_sum_f64(s->comm, agree_dev, 1, s->stream));
            GP_CUDA(cudaMemcpyAsync(&short_all, agree_dev, sizeof(double), cudaMemcpyDeviceToHost, s->stream));
            GP_CUDA(cudaStreamSynchronize(s->stream));
        }
        if (short_all != 0.0) {
            set_last_error("IRF bands at level %g over %d sampling iterations need %.0f bytes of device memory for their tail "
                           "buffers (%.0f in all); %zu bytes are free on this device%s", irf->band, S, tail_bytes,
                           need, free_b, need > (double)free_b ? "" : " (another rank lacks them)");
            return GPIRT_B200_ERR_NOMEM;
        }
        const cudaError_t e = cudaMalloc((void**)&irf_buf, (size_t)need);
        if (e != cudaSuccess) {
            cudaGetLastError();
            irf_buf = nullptr;
            set_last_error("device allocation of %.0f bytes for the IRF summaries failed: %s", need, cudaGetErrorString(e));
            return GPIRT_B200_ERR_NOMEM;
        }
        irf->band_bytes = (int64_t)tail_bytes;
        if (irf_bands) {
            irf_lo = irf_buf + 2 * irf_plane;
            irf_hi = irf_lo + (size_t)irf_plan.klo * irf_plane;
        }
        if (fs_out) {
            for (int i = 0; i < 2; ++i) GP_TRY(pool_alloc((void**)&snap_fs[i], irf_plane * sizeof(double), s->stream));
            // pinned bounce buffers large enough for an f* plane now: the storage worker must never reallocate them while
            // the other buffer's transfer is in flight (without pinned memory the plane goes by a plain copy)
            bo->ensure(std::max(keep_f ? nm : (size_t)0, irf_plane));
        }
    }
    // posterior predictive checks: the chi-square counters from the pool; the pair state (observed counts of every pair,
    // counters, replicate plane) in one cudaMalloc, checked against the free device memory before the first sweep, and
    // the observed counts computed now
    if (ppc) {
        ppc->ppp = NAN;
        ppc->pair_bytes = 0;
        GP_TRY(ppc_chi2.init(s->stream, s->y8, s->ldy8, (int)n, (int)m));
        if (ppc->pair_ppp || ppc->pair_log_or) {
            const double need = (double)PpcPairs::bytes_needed(n, m, s->has_missing);
            ppc->pair_bytes = (int64_t)need;   // also reported when the call is refused
            size_t free_b = 0;
            GP_TRY(free_memory_for(need, s->stream, &free_b));
            if (need > (double)free_b) {
                set_last_error("the pair checks of %lld items over %lld respondents need %.0f bytes of device memory; %zu bytes "
                               "are free on this device", (long long)m, (long long)n, need, free_b);
                return GPIRT_B200_ERR_NOMEM;
            }
            GP_TRY(ppc_pairs.init(s->stream, s->y8, s->ldy8, (int)n, (int)m, s->has_missing));
        }
    }
    t_c = now();
    GP_TRY(s->init_draws());
    t_d = now();
    // drain(slot), on the storage worker: the copy stream waits for the snapshot, then the worker blocks in the
    // device-to-host copies.  The sampler's status words (Cholesky / ESS failure) ride along, so a failed chain is noticed
    // at the next stored slot instead of spinning every item through the ESS iteration cap for the rest of the run.
    worker = new StoreWorker();
    GP_CUDA(cudaGetDevice(&worker->device));
    // issue(slot): the copy stream waits for the snapshot and gets every device-to-host transfer of the slot (status words,
    // theta | beta into pinned staging, f in pieces into the pinned bounce buffer); finish(slot): the host copies.
    // The worker issues slot k+1 (other snapshot / bounce / staging buffers) before it finishes slot k, so the PCIe transfer
    // of one slice runs under the host copies of the previous one.
    worker->issue = [this](int slot) -> int {            // theta_draws.row(slot), beta_draws.slice(slot), f_draws.slice(slot)
        const int b = slot & 1;
        GP_CUDA(cudaStreamWaitEvent(copy, ev[b], 0));
        GP_CUDA(cudaMemcpyAsync((void*)w_poll, s->status, 4 * sizeof(int), cudaMemcpyDeviceToHost, copy));
        GP_CUDA(cudaMemcpyAsync(h_small[b], snap_small[b], n_small * sizeof(double), cudaMemcpyDeviceToHost, copy));
        GP_CUDA(cudaEventRecord(ev_small[b], copy));
        if (keep_f) GP_TRY(bounce_issue(*bo, copy_threads, f_out + (size_t)slot * nm, snap_f[b], nm, b, copy, xfer[b]));
        return GPIRT_B200_OK;
    };
    worker->finish = [this](int slot) -> int {
        const double ts0 = now();
        const int b = slot & 1;
        if (keep_f) GP_TRY(bounce_finish(b, xfer[b]));
        GP_CUDA(cudaEventSynchronize(ev_small[b]));
        const double* small = h_small[b];
        for (int64_t i = 0; i < n; ++i) theta_out[(size_t)i * n_slots + slot] = small[i];
        std::memcpy(beta_out + (size_t)slot * 2 * m, small + n, 2 * (size_t)m * sizeof(double));
        if (fs_out) {   // the f* plane after this slot's f slice, through the same bounce buffer (its DMA has landed)
            double* dst = fs_out + (size_t)slot * irf_plane;
            if (irf_plane <= bo->cap) GP_TRY(d2h(dst, snap_fs[b], irf_plane, b));
            else {
                GP_CUDA(cudaMemcpyAsync(dst, snap_fs[b], irf_plane * sizeof(double), cudaMemcpyDeviceToHost, copy));
                GP_CUDA(cudaStreamSynchronize(copy));
            }
        }
        worker->busy_s += now() - ts0;
        return GPIRT_B200_OK;
    };
    worker->start();
    GP_TRY(snapshot(0));                                                            // :53-55 initial values
    worker->push(0);
    return GPIRT_B200_OK;
}

int ChainRun::iterate(int iter) {
    const bool sampling = iter >= B;
    const int si = iter - B + 1;                                                    // 1-based sampling iteration
    const bool store = sampling && si % thin == 0;
    GP_TRY(s->sweep(sampling ? 1 : 0));                                             // enqueue sweep (asynchronous)
    if (sampling && summarise_f) {
        dim3 grid((unsigned)m, (unsigned)ceil_div(n, 256));
        GP_LAUNCH(k_f_welford, grid, 256, 0, s->stream, s->f, s->ldn, (int)n, (double)(++n_summarised), f_mean, f_m2);
    }
    if (sampling && fit)
        GP_TRY(launch_predictive_accumulate(s->stream, s->f, s->ldn, pred_code, s->ldy8, s->theta, s->beta, (int)n, (int)m,
                                            (double)si, pred_acc));
    if (sampling && irf)   // the f* this sweep drew (fstar, not the means in Dmat); nothing on a side stream writes it
        GP_TRY(launch_irf_accumulate(s->stream, s->fstar, s->ldN, N_GRID, irf_cells, si, irf_buf, irf_buf + irf_plane,
                                     irf_lo, irf_plan.klo, irf_hi, irf_plan.khi));
    if (sampling && ppc) {   // the replicate of the state this sweep left, under the counter of that sweep (B + si)
        GP_TRY(ppc_chi2.iterate(s->stream, s->f, s->ldn, s->y8, s->ldy8, s->theta, s->beta, s->key_at(s->sweep_counter),
                                s->item_offset, ppc_pairs.buf ? ppc_pairs.yrep : nullptr));
        if (ppc_pairs.buf) GP_TRY(ppc_pairs.iterate(s->stream));
    }
    if (sampling && (diag_trace || diag_halves))   // theta | beta as the snapshot would copy them, and f* as above
        GP_TRY(launch_chain_halves(s->stream, s->fstar, s->ldN, N_GRID, irf_cells, si, S, diag_halves, s->theta, (int)n,
                                   s->beta, 2 * (int)m, diag_trace));
    if (store) {
        const int slot = si / thin;                                                 // :99-103
        worker->wait_buffer_free(slot & 1);                                         // slot - 2 has left this snapshot buffer
        GP_TRY(snapshot(slot));
        worker->push(slot);
    }
    if ((iter & 7) == 7) {                                                          // bounded run-ahead; progress / interrupts stay honest
        GP_TRY(enqueue_agreement());
        GP_CUDA(cudaMemcpyAsync(h_poll, s->status, 4 * sizeof(int), cudaMemcpyDeviceToHost, s->stream));
        GP_CUDA(cudaStreamSynchronize(s->stream));
        if (stop_now(agree_count - 1)) return stop_code;
    }
    return GPIRT_B200_OK;
}

int ChainRun::finish() {
    worker->wait_idle();
    const double t_store = worker->busy_s;
    {
        std::string msg;
        const int wrc = worker->status(&msg);
        if (wrc != GPIRT_B200_OK) { set_last_error("%s", msg.c_str()); return wrc; }
    }
    GP_CUDA(cudaMemcpyAsync(h_poll, s->status, 4 * sizeof(int), cudaMemcpyDeviceToHost, s->stream));
    GP_CUDA(cudaStreamSynchronize(s->stream));
    if (!sharded && stop_now(-1)) return stop_code;
    GP_TRY(s->check_status());
    {
        int h[4] = {0, 0, 0, 0};
        GP_CUDA(cudaMemcpy(h, s->status, sizeof(h), cudaMemcpyDeviceToHost));
        degenerate = h[2];   // theta draws whose CDF was degenerate (grid point 0 taken; the reference reads out of bounds there)
    }
    // IRFs = plogis(IRFs / S)   (:106-111; S = 0 gives NaN exactly as the reference's 0 * inf)
    const double inv = 1.0 / (double)S;
    GP_TRY(launch_irf_finish(s->stream, s->irf_sum, s->ldN, N_GRID, (int)m, inv, s->Dmat));
    GP_CUDA(cudaMemcpyAsync(irf_out, s->Dmat, (size_t)N_GRID * m * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
    if (summarise_f) {
        if (n_summarised == 0) {
            GP_CUDA(cudaMemsetAsync(f_mean, 0xff, nm * sizeof(double), s->stream));   // all-ones bit pattern = NaN: no sampling iterations
            GP_CUDA(cudaMemsetAsync(f_m2, 0xff, nm * sizeof(double), s->stream));
        } else {
            GP_LAUNCH(k_f_sd, (unsigned)ceil_div((int64_t)nm, 256), 256, 0, s->stream, f_m2, nm, (double)(n_summarised - 1));
        }
        // fresh pageable destinations: the chunked pinned-bounce copy with host threads, as for the f draws
        GP_CUDA(cudaStreamSynchronize(s->stream));
        if (f_mean_out) GP_TRY(d2h(f_mean_out, f_mean, nm, 0));
        if (f_sd_out) GP_TRY(d2h(f_sd_out, f_m2, nm, 1));
    }
    if (fit) {
        const double Sd = (double)S;
        if (S == 0) {   // NaN accumulators: every output NaN, the cell counts still hold
            GP_CUDA(cudaMemsetAsync(pred_acc, 0xff, pred_plane * sizeof(double), s->stream));
            GP_CUDA(cudaMemsetAsync(pred_acc + 2 * pred_plane, 0xff, pred_plane * sizeof(double), s->stream));
        }
        GP_TRY(launch_predictive_reduce(s->stream, pred_acc, s->ldn, pred_code, s->ldy8, (int)n, (int)m, Sd, pred_stats,
                                        pred_partial, PRED_CHUNKS, pred_resp));
        if (sharded) GP_TRY(comm_allreduce_sum_f64(s->comm, pred_resp, (size_t)n + PRED_STATS, s->stream));
        double tot[PRED_STATS];
        GP_CUDA(cudaMemcpyAsync(tot, pred_resp + n, sizeof(tot), cudaMemcpyDeviceToHost, s->stream));
        if (fit->elpd_resp) GP_CUDA(cudaMemcpyAsync(fit->elpd_resp, pred_resp, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
        if (fit->elpd_item) GP_CUDA(cudaMemcpyAsync(fit->elpd_item, pred_stats + 2 * (size_t)m, (size_t)m * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
        // per-cell outputs one at a time, tightly packed into the (now free) running-mean plane
        double* const outs[3] = {fit->pred, fit->lpd_cell, fit->pwaic_cell};
        for (int w = 0; w < 3; ++w) {
            if (!outs[w]) continue;
            GP_TRY(launch_predictive_cells(s->stream, pred_acc, s->ldn, pred_code, s->ldy8, (int)n, (int)m, Sd, w, pred_acc + pred_plane));
            GP_CUDA(cudaStreamSynchronize(s->stream));
            GP_TRY(d2h(outs[w], pred_acc + pred_plane, nm, 0));
        }
        GP_CUDA(cudaStreamSynchronize(s->stream));
        const double N = tot[5], sum_e = tot[2], var = (tot[3] - sum_e * sum_e / N) / (N - 1.0);
        fit->lppd = tot[0];
        fit->p_waic = tot[1];
        fit->elpd_waic = tot[0] - tot[1];
        fit->waic = -2.0 * fit->elpd_waic;
        fit->se_elpd_waic = std::sqrt(N * (var < 0.0 ? 0.0 : var));   // loo's convention; NaN stays NaN
        fit->lpd_holdout = S ? tot[4] : NAN;   // S = 0: NaN even where no cell is held out
        fit->n_obs = (int64_t)tot[5];
        fit->n_holdout = (int64_t)tot[6];
    }
    if (irf) {
        double* const mean = irf_buf;
        double* const m2 = mean + irf_plane;
        if (S == 0) {   // all-ones bit pattern = NaN: no sampling iterations
            GP_CUDA(cudaMemsetAsync(mean, 0xff, 2 * irf_plane * sizeof(double), s->stream));
        } else {   // sd over M2 in place; the band ends over heap slot 0 of each heap (read before written, per cell)
            GP_TRY(launch_irf_finish_bands(s->stream, irf_cells, S, m2, m2, irf_lo, irf_hi, irf_plan, true,
                                           irf_lo, irf_hi));
        }
        GP_CUDA(cudaStreamSynchronize(s->stream));
        if (irf->prob_mean) GP_TRY(d2h(irf->prob_mean, mean, irf_plane, 0));
        if (irf->prob_sd) GP_TRY(d2h(irf->prob_sd, m2, irf_plane, 1));
        if (irf->lower) GP_TRY(d2h(irf->lower, irf_bands ? irf_lo : m2, irf_plane, 0));   // S = 0: the NaN plane
        if (irf->upper) GP_TRY(d2h(irf->upper, irf_bands ? irf_hi : m2, irf_plane, 1));
    }
    if (ppc) {
        GP_TRY(ppc_chi2.finish(s->stream, S, ppc->item_ppp, ppc->resp_ppp, &ppc->ppp));
        auto copy = [this](double* dst, const double* src, size_t count) { return d2h(dst, src, count, 0); };
        if (ppc_pairs.buf) GP_TRY(ppc_pairs.finish(s->stream, 1.0 / (double)S, S == 0, ppc->pair_log_or, ppc->pair_ppp, copy));
    }
    GP_CUDA(cudaStreamSynchronize(s->stream));
    if (trace)
        fprintf(stderr, "gpirt_b200_mcmc: create %.3fs, copy buffers %.3fs, init draws %.3fs, %d sweeps + stores %.3fs (stores %.3fs)\n",
                t_b - t_a, t_c - t_b, t_d - t_c, S + B, now() - t_d, t_store);
    return GPIRT_B200_OK;
}

// Several chains in one call (opts.chains): C ChainRuns on the current device, each with its own seed, sampler, streams,
// graph, snapshot buffers and storage worker; this thread enqueues sweep t of chain 0, 1, ..., C - 1 in turn, so no two
// chains' graph captures interleave.  Diagnostics over all S sampling iterations on the device (k_chain_diag,
// k_chain_irf_rhat) after the last sweep.
int mcmc_chains(const double* y, int64_t n, int64_t m, const double* theta_init, int S, int B, const double* pm,
                const double* psd, const double* pstep, const gpirt_b200_opts* opts, double* theta_out, double* beta_out,
                double* f_out, double* irf_out, gpirt_b200_progress_cb cb, void* cb_ctx, bool trace) {
    gpirt_b200_chains* const ch = opts->chains;
    ch->diag_bytes = 0;
    const int C = ch->chains;
    if (C < 1 || C > 32) { set_last_error("bad argument: chains must lie in [1, 32], got %d", C); return GPIRT_B200_ERR_ARG; }
    if (opts->world_size > 1) { set_last_error("several chains with items sharded across GPUs are not built"); return GPIRT_B200_ERR_ARG; }
    if (opts->fit || opts->irf || opts->ppc || opts->f_mean_out || opts->f_sd_out) {
        set_last_error("fit, irf, ppc, f_mean_out and f_sd_out are not built for several chains");
        return GPIRT_B200_ERR_ARG;
    }
    if (!theta_init) { set_last_error("bad argument: theta_init is NULL"); return GPIRT_B200_ERR_ARG; }
    const bool want_diag = ch->theta_rhat || ch->theta_ess || ch->beta_rhat || ch->beta_ess;
    const bool diag_on = S >= 4;                          // fewer iterations: every diagnostic is NaN
    const int64_t P = n + 2 * m, cells = (int64_t)N_GRID * m;
    const size_t trace_elems = want_diag && diag_on ? (size_t)S * P * C : 0;
    const size_t halves_elems = ch->irf_rhat && diag_on ? (size_t)4 * cells * C : 0;
    const size_t out_elems = (trace_elems ? 2 * (size_t)P : 0) + (halves_elems ? (size_t)cells : 0);
    ch->diag_bytes = (int64_t)((trace_elems + halves_elems) * sizeof(double));
    const int threads = host_threads_for_copy(C);
    int dev = 0;
    if (opts->device >= 0) GP_CUDA(cudaSetDevice(opts->device));
    GP_CUDA(cudaGetDevice(&dev));
    cudaMemPool_t pool;
    GP_CUDA(cudaDeviceGetDefaultMemPool(&pool, dev));
    // Destroyed last: the diagnostics buffer is freed, and with C > 1 the pool is trimmed so that C samplers' memory does
    // not stay reserved on a shared device after the call.
    struct CallEnd {
        int C; cudaMemPool_t pool; double* diag = nullptr;
        ~CallEnd() {
            if (diag) cudaFree(diag);
            if (C > 1) { cudaDeviceSynchronize(); cudaMemPoolTrimTo(pool, 0); }
        }
    } end{C, pool};
    if (C > 1) { GP_CUDA(cudaDeviceSynchronize()); GP_CUDA(cudaMemPoolTrimTo(pool, 0)); }
    struct OwnBounces {                                   // pinned staging of chains 1..C-1 (chain 0: g_bounce)
        std::unique_ptr<Bounce[]> b;
        int C;
        ~OwnBounces() {
            for (int c = 1; c < C; ++c) {
                b[c].release();
                for (auto& v : b[c].ev) for (cudaEvent_t e : v) cudaEventDestroy(e);
            }
        }
    } own{std::unique_ptr<Bounce[]>(new Bounce[C]), C};
    std::vector<gpirt_b200_opts> copt(C, *opts);
    std::vector<std::unique_ptr<ChainRun>> runs;
    for (int c = 0; c < C; ++c) {
        copt[c].seed = ch->seeds ? ch->seeds[c] : opts->seed + (uint64_t)c;
        copt[c].chains = nullptr;
        const size_t slots = (size_t)((opts->thin > 1 ? S / opts->thin : S) + 1);
        runs.emplace_back(new ChainRun{y, n, m, theta_init + (size_t)c * n, S, B, pm, psd, pstep, &copt[c],
                                       theta_out + (size_t)c * slots * n, beta_out + (size_t)c * 2 * m * slots,
                                       f_out ? f_out + (size_t)c * slots * n * m : nullptr, irf_out + (size_t)c * cells,
                                       c == 0 ? &g_bounce : &own.b[c], threads, trace && c == 0});
        runs[c]->untraced = c > 0;
    }
    auto failed = [&](int c, int rc) {
        const std::string msg = last_error();
        set_last_error("chain %d: %s", c, msg.c_str());
        return rc;
    };
    // Memory, before the first sweep: chain 0's footprint is the drop of free device memory across its set-up; the other
    // chains and the diagnostics must fit in what is left.
    size_t free0 = 0, free1 = 0, total = 0;
    GP_CUDA(cudaMemGetInfo(&free0, &total));
    if (int rc = runs[0]->setup()) return failed(0, rc);
    GP_CUDA(cudaStreamSynchronize(runs[0]->s->stream));
    GP_CUDA(cudaMemGetInfo(&free1, &total));
    const double footprint = free0 > free1 ? (double)(free0 - free1) : 0.0;
    const double need = (C - 1) * footprint + (double)(trace_elems + halves_elems + out_elems) * sizeof(double);
    if (need > (double)free1) {
        set_last_error("%d chains need %.0f more bytes of device memory (%.0f per further chain, %lld for the diagnostics); "
                       "%zu bytes are free on this device", C, need, footprint, (long long)ch->diag_bytes, free1);
        return GPIRT_B200_ERR_NOMEM;
    }
    double *trace_dev = nullptr, *halves_dev = nullptr, *out_dev = nullptr;
    if (const size_t elems = trace_elems + halves_elems + out_elems) {
        const cudaError_t e = cudaMalloc((void**)&end.diag, elems * sizeof(double));
        if (e != cudaSuccess) {
            cudaGetLastError();
            end.diag = nullptr;
            set_last_error("device allocation of %zu bytes for the chain diagnostics failed: %s", elems * sizeof(double), cudaGetErrorString(e));
            return GPIRT_B200_ERR_NOMEM;
        }
        trace_dev = trace_elems ? end.diag : nullptr;
        halves_dev = halves_elems ? end.diag + trace_elems : nullptr;
        out_dev = end.diag + trace_elems + halves_elems;
    }
    for (int c = 0; c < C; ++c) {
        if (trace_dev) runs[c]->diag_trace = trace_dev + (size_t)c * P * S;
        if (halves_dev) runs[c]->diag_halves = halves_dev + (size_t)c * 4 * cells;
        if (c > 0) if (int rc = runs[c]->setup()) return failed(c, rc);
    }
    const int total_it = S + B;
    const double inc = total_it > 0 ? 100.0 / total_it : 0.0;
    double progress = 0.0;
    for (int iter = 0; iter < total_it; ++iter) {
        if (cb && cb(progress, cb_ctx)) for (auto& r : runs) r->want_stop = true;   // Rcpp::checkUserInterrupt, :66,85
        for (int c = 0; c < C; ++c) if (runs[c]->stopped()) return failed(c, runs[c]->stop_code);
        progress += inc;
        for (int c = 0; c < C; ++c) if (int rc = runs[c]->iterate(iter)) return failed(c, rc);
    }
    int64_t degenerate = 0;
    for (int c = 0; c < C; ++c) {
        const int rc = runs[c]->finish();
        degenerate += runs[c]->degenerate;
        g_last_degenerate_theta = degenerate;
        if (rc != GPIRT_B200_OK) return failed(c, rc);
    }
    // every chain's stream has drained (finish): the diagnostics run on chain 0's
    cudaStream_t st = runs[0]->s->stream;
    auto put = [&](double* dst, const double* src, size_t count) -> int {
        if (!dst) return GPIRT_B200_OK;
        if (!src) { std::fill(dst, dst + count, (double)NAN); return GPIRT_B200_OK; }
        GP_CUDA(cudaMemcpyAsync(dst, src, count * sizeof(double), cudaMemcpyDeviceToHost, st));
        return GPIRT_B200_OK;
    };
    double *rhat_dev = nullptr, *ess_dev = nullptr, *irf_rhat_dev = nullptr;
    if (trace_dev) {
        rhat_dev = out_dev;
        ess_dev = out_dev + P;
        GP_TRY(launch_chain_diag(st, trace_dev, (int)P, S, C, rhat_dev, ess_dev));
    }
    if (halves_dev) {
        irf_rhat_dev = out_dev + (trace_dev ? 2 * P : 0);
        GP_TRY(launch_chain_irf_rhat(st, halves_dev, cells, S, C, irf_rhat_dev));
    }
    GP_TRY(put(ch->theta_rhat, rhat_dev, (size_t)n));
    GP_TRY(put(ch->theta_ess, ess_dev, (size_t)n));
    GP_TRY(put(ch->beta_rhat, rhat_dev ? rhat_dev + n : nullptr, 2 * (size_t)m));
    GP_TRY(put(ch->beta_ess, ess_dev ? ess_dev + n : nullptr, 2 * (size_t)m));
    GP_TRY(put(ch->irf_rhat, irf_rhat_dev, (size_t)cells));
    GP_CUDA(cudaStreamSynchronize(st));
    if (cb) cb(100.0, cb_ctx);
    return GPIRT_B200_OK;
}
}  // namespace

int gpirt_b200_mcmc(const double* y, int64_t n, int64_t m, const double* theta_init, int sample_iterations,
                    int burn_iterations, const double* pm, const double* psd, const double* pstep,
                    const gpirt_b200_opts* opts, double* theta_out, double* beta_out, double* f_out, double* irf_out,
                    gpirt_b200_progress_cb cb, void* cb_ctx) {
    if (sample_iterations < 0 || burn_iterations < 0 || !theta_out || !beta_out || !irf_out) {
        set_last_error("bad argument: negative iteration count or null output");
        return GPIRT_B200_ERR_ARG;
    }
    const bool keep_f = !(opts && opts->skip_f_draws);
    if (keep_f && !f_out) { set_last_error("f_out is NULL but f draws were requested"); return GPIRT_B200_ERR_ARG; }
    if (opts && opts->thin < 0) { set_last_error("bad argument: thin < 0"); return GPIRT_B200_ERR_ARG; }
    gpirt_b200_irf* const irf = opts ? opts->irf : nullptr;
    if (irf && (irf->lower || irf->upper) && !(std::isfinite(irf->band) && irf->band > 0.0 && irf->band < 1.0)) {
        set_last_error("bad argument: the IRF band level must lie in (0, 1), got %g", irf->band);
        return GPIRT_B200_ERR_ARG;
    }
    if (opts && opts->ppc && opts->world_size > 1) {   // every rank sees its own opts: all refuse before any collective
        set_last_error("posterior predictive checks with items sharded across GPUs are not built");
        return GPIRT_B200_ERR_ARG;
    }
    const bool trace = getenv("GPIRT_TIMING") != nullptr;
    g_last_degenerate_theta = 0;
    struct ExitTrace {   // first local: destroyed last
        bool on; double t_enter; double t_body_end = 0.0;
        ~ExitTrace() {
            if (!on) return;
            const double t = ChainRun::now();
            fprintf(stderr, "gpirt_b200_mcmc: total %.3fs in the call, %.3fs after the body\n", t - t_enter, t_body_end > 0.0 ? t - t_body_end : 0.0);
        }
    } exit_trace{trace, ChainRun::now()};
    // the pinned bounce buffers are process-wide: a call that moves f through them owns them until it returns
    std::unique_lock<std::mutex> bounce_lock(g_bounce_mu);
    if (opts && opts->chains) {
        const int rc = mcmc_chains(y, n, m, theta_init, sample_iterations, burn_iterations, pm, psd, pstep, opts, theta_out,
                                   beta_out, f_out, irf_out, cb, cb_ctx, trace);
        exit_trace.t_body_end = ChainRun::now();
        return rc;
    }
    ChainRun run{y, n, m, theta_init, sample_iterations, burn_iterations, pm, psd, pstep, opts, theta_out, beta_out, f_out,
                 irf_out, &g_bounce, host_threads_for_copy(1), trace};
    GP_TRY(run.setup());
    const int total = sample_iterations + burn_iterations;
    const double inc = total > 0 ? 100.0 / total : 0.0;
    double progress = 0.0;
    for (int iter = 0; iter < total; ++iter) {
        if (cb && cb(progress, cb_ctx)) run.want_stop = true;                      // Rcpp::checkUserInterrupt, :66,85
        if (run.stopped()) return run.stop_code;
        progress += inc;
        GP_TRY(run.iterate(iter));
    }
    const int rc = run.finish();
    g_last_degenerate_theta = run.degenerate;
    if (rc != GPIRT_B200_OK) return rc;
    if (cb) cb(100.0, cb_ctx);
    exit_trace.t_body_end = ChainRun::now();
    return GPIRT_B200_OK;
}

}  // extern "C"
