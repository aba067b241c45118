// qlnlp.cu -- C ABI (include/qlnlp.h) over the fused evaluator kernel, plus the host-side planner
// (segment plan, Jacobian structure, bounds) and the host-pointer pipeline.  Built with nvcc for sm_100a only;
// no CPU fallback: every evaluation entry point runs the CUDA kernels or fails.
#include "../../include/qlnlp.h"

#include <cuda.h>
#include <cudaTypedefs.h>
#include <cuda_runtime.h>
#include <sys/mman.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <climits>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <initializer_list>
#include <map>
#include <memory>
#include <mutex>
#include <new>
#include <string>
#include <tuple>
#include <type_traits>
#include <utility>
#include <vector>

#include "hostrows.h"
#include "layout.h"
#include "qlnlp_hess.cuh"
#include "qlnlp_kin.cuh"
#include "qlnlp_kkt.cuh"

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CUDA_TRY(expr)                                                                              \
    do {                                                                                            \
        cudaError_t e_ = (expr);                                                                    \
        if (e_ != cudaSuccess)                                                                      \
            return fail(e_ == cudaErrorMemoryAllocation ? QLNLP_ENOMEM : QLNLP_ECUDA, "%s: %s (%s:%d)", #expr, \
                        cudaGetErrorString(e_), __FILE__, __LINE__);                                \
    } while (0)

// Owners of what a handle holds on the device.  device_alloc / pinned_alloc count a block in, its deleter counts it out.
std::atomic<int> g_owned_blocks{0};
std::atomic<int64_t> g_fail_alloc{-1};  // tests: allocations to go before one fails as out of memory (negative: none)
struct CudaFree { void operator()(void* p) const { cudaFree(p); --g_owned_blocks; } };
struct CudaFreeHost { void operator()(void* p) const { cudaFreeHost(p); --g_owned_blocks; } };
struct StreamDestroy { void operator()(cudaStream_t s) const { cudaStreamDestroy(s); } };
struct EventDestroy { void operator()(cudaEvent_t e) const { cudaEventDestroy(e); } };
template <typename T> using DevPtr = std::unique_ptr<T, CudaFree>;
template <typename T> using PinnedPtr = std::unique_ptr<T, CudaFreeHost>;
using Stream = std::unique_ptr<std::remove_pointer_t<cudaStream_t>, StreamDestroy>;
using Event = std::unique_ptr<std::remove_pointer_t<cudaEvent_t>, EventDestroy>;

// A failed allocation, mapped as CUDA_TRY maps it; an out-of-memory must not linger as the thread's last error.
int alloc_failed(cudaError_t e, const char* what, size_t bytes)
{
    cudaGetLastError();
    return fail(e == cudaErrorMemoryAllocation ? QLNLP_ENOMEM : QLNLP_ECUDA, "%s of %zu bytes: %s", what, bytes,
                cudaGetErrorString(e));
}

template <typename T>
int device_alloc(DevPtr<T>& out, size_t n)
{
    void* p = nullptr;
    const cudaError_t e = g_fail_alloc.fetch_sub(1) == 0 ? cudaErrorMemoryAllocation : cudaMalloc(&p, sizeof(T) * n);
    if (e != cudaSuccess) return alloc_failed(e, "cudaMalloc", sizeof(T) * n);
    ++g_owned_blocks;
    out.reset(static_cast<T*>(p));
    return QLNLP_OK;
}

template <typename T>
int pinned_alloc(PinnedPtr<T>& out, size_t n, unsigned flags)
{
    void* p = nullptr;
    const cudaError_t e = g_fail_alloc.fetch_sub(1) == 0 ? cudaErrorMemoryAllocation : cudaHostAlloc(&p, sizeof(T) * n, flags);
    if (e != cudaSuccess) return alloc_failed(e, "cudaHostAlloc", sizeof(T) * n);
    ++g_owned_blocks;
    out.reset(static_cast<T*>(p));
    return QLNLP_OK;
}

// A device copy of n values, handed to `out` only once complete: a table is either absent or valid.  The copy may still
// be in flight when cudaMemcpy returns (pageable source) and launches go to any stream, so `sync` waits for the device
// before the hand-over; a set-up of several tables waits once, after the last.
template <typename T>
int upload(DevPtr<T>& out, const T* src, size_t n, bool sync = true)
{
    DevPtr<T> d;
    if (int rc = device_alloc(d, n)) return rc;
    CUDA_TRY(cudaMemcpy(d.get(), src, sizeof(T) * n, cudaMemcpyHostToDevice));
    if (sync) CUDA_TRY(cudaDeviceSynchronize());
    out = std::move(d);
    return QLNLP_OK;
}

constexpr int TICKET_POOL = 64;       // work counters of streams (recycled once every one is taken)
constexpr int GRAPH_TICKETS = 1024;   // work counters of captured graphs (each held until its graph is destroyed)
constexpr int NJM = 4;                 // kernel value streams: JM_NONE, JM_BLOCK, JM_TRUE, JM_VALS
constexpr int MAX_LANES = 4;           // pipeline depth of the host-pointer path
constexpr int64_t COMPACT_MIN_B = 64;  // below this, host-pointer batches copy the pattern rows as they are

// Every entry point that touches the device makes the handle's device current and restores the caller's on exit
// (a multi-GPU host -- torch, CUDA.jl -- must not find its current device changed by a call into this library).
struct DeviceGuard {
    int prev = -1, dev;
    explicit DeviceGuard(int d) : dev(d)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) cudaSetDevice(dev);
    }
    ~DeviceGuard()
    {
        if (prev >= 0 && prev != dev) cudaSetDevice(prev);
    }
};

// per-stream scratch of the host-pointer pipeline
struct HostLane {
    Stream stream;
    Event done;                 // the chunk's last copy has landed
    int64_t cap = 0;            // evaluations the buffers hold
    DevPtr<double> Z, x0, xf, f, grad, g, jac;
    PinnedPtr<double> stage;    // host rows of VALS values awaiting the row builder
};

// device memory that only grows (per-stream scratch, single-call slots)
struct Scratch {
    DevPtr<double> ptr;
    size_t cap = 0;             // doubles
};

// single evaluations (the four MOI callbacks): one launch per decision vector, results cached
struct OneEval {
    Stream stream;
    Scratch slots;              // device rows of the other single calls (single_call)
    PinnedPtr<double> hx;       // mapped: x(ldz_e) | f(2) grad(ldgrad_e) g(ldg_e) vals(ldv_e)
    double* hout = nullptr;
    double* mx = nullptr;       // device-side addresses of hx / hout: the kernel reads x and writes the results there
    double* mout = nullptr;
    int64_t o_grad = 0, o_g = 0, o_vals = 0, total = 0;
    bool valid = false;         // hout holds the results for the x stored in hx
};

struct Registration {
    double* ptr;
    int64_t ld, rows;
};

// class table of a ragged launch (device copy of one QlRagClass per handle)
struct RagTable {
    DevPtr<unsigned char> d_classes;   // QL_RAGCLASS_BYTES per class
    QlClass layout;                    // the class with the largest N: sizes the shared-memory carve-up
    bool fastdiv = false;
};

// One SPARSE_BLOCK value of the block plan (block_plan)
struct BlockEntry {
    int32_t row, col;                  // 1-based
    double konst;                      // the constant image: what the value is where it does not depend on Z, else 0
    bool vals;                         // depends on Z: part of the VALS stream
};

// The problem a handle evaluates: built once when the handle is created, host memory only, read-only afterwards.
struct Problem {
    QlClass cls;
    int jac_mode = QLNLP_JAC_SPARSE_BLOCK;
    // opt-in kinematic rows (qlnlp_kin.cuh): 2N more constraints, 8N more entries in either sparse pattern
    bool kin = false;
    double leg_reach = 0;              // l1 + l2 + lb/2
    double x0xf[2 * QL_NX];            // x0 | xf
    std::vector<double> cost;          // field-major [QL_NCOST][npad]
    int npad = 0;
    std::vector<BlockEntry> block;     // every SPARSE_BLOCK value in value order: the one source of every host pattern table
    std::vector<QlSeg> segs;
    std::vector<int> seg_begin;
    double rmb = 0, rmf = 0, rIb = 0;  // reciprocals of the divisors
    bool fastdiv = false;              // reciprocal-FMA division verified exact for this model
    uint64_t serial = 0;               // unique per handle ever created (addresses get reused)
    int64_t ldz_e = 0, ldgrad_e = 0, ldg_e = 0, ldjac_e = 0, ldv_e = 0;   // even leading dimensions of the scratch
};

// Work counters that captured graphs own: the GRAPH_TICKETS counters after the stream pool.  A capture sequence takes
// one per stream at its first launch there, and its graph holds it through a CUDA user object until the graph (and
// every executable instantiated from it) is destroyed.  The user object's destructor runs on a thread of the CUDA
// runtime, may make no CUDA call and may run after the handle is gone: it only hands the counter back, under `mu`.
struct GraphTickets {
    std::mutex mu;
    std::vector<int> free;                                                // counters no graph holds
    std::map<std::pair<unsigned long long, cudaStream_t>, int> live;     // (capture sequence, stream) -> counter
};

struct GraphTicket {
    std::shared_ptr<GraphTickets> pool;
    std::pair<unsigned long long, cudaStream_t> key;
    int index;
};

void release_graph_ticket(void* p)
{
    std::unique_ptr<GraphTicket> t(static_cast<GraphTicket*>(p));
    std::lock_guard<std::mutex> lk(t->pool->mu);
    t->pool->live.erase(t->key);
    t->pool->free.push_back(t->index);        // zero again: the last CTA of every grid re-arms its counter
}

// What one device of a handle holds, created at its first evaluation (ensure_device).
struct DeviceState {
    int device = 0;
    bool ready = false;
    std::string pci_bus_id;
    int sm_count = 0;
    size_t smem_per_sm = 0, smem_optin = 0;
    std::map<std::pair<const void*, size_t>, int> blocks_per_sm;   // (kernel, dynamic smem) -> resident CTAs (kernel_geometry)
    DevPtr<double> d_cost;
    DevPtr<double> d_x0xf;             // x0[15] | xf[15]
    DevPtr<QlSeg> d_segs;
    DevPtr<int> d_seg_begin;
    DevPtr<long long> d_dense_lin;     // DENSE mode: linear index of every SPARSE_BLOCK value
    HostLane lanes[MAX_LANES];
    OneEval one;
    std::map<cudaStream_t, unsigned*> tickets;   // work counters, one pair per stream the device has launched on
    DevPtr<unsigned> ticket_pool;                // pre-zeroed counters (128 B apart) so that a launch needs no
    int ticket_pool_used = 0;                    // allocation: launches stay legal inside CUDA-graph capture
    std::shared_ptr<GraphTickets> graph_tickets; // the counters after the TICKET_POOL stream counters
    DevPtr<int> d_kin_map;             // caller-visible value order of the batch pattern -> scratch position or -(entry + 1)
    std::map<cudaStream_t, Scratch> kin_scratch;                 // per stream: reference-order rows (device)
    std::map<std::vector<uint64_t>, RagTable> rag_tables;       // ragged launches led by this handle (key: the classes' serials)
    DevPtr<unsigned short> d_kkt_tab;  // KKT solve: slot / column of every SPARSE_TRUE value, then row / column of every W value
    std::map<cudaStream_t, Scratch> kkt_scratch;                 // per stream: factor scratch of every resident warp
    int64_t last_launch[5] = {0, 0, 0, 0, 0};
    std::unique_ptr<qlhost::Pool> pool;                                  // row builders of the host-pointer path
    int64_t stat_host_rows = 0, stat_host_lines = 0;                     // rows / 64-byte lines the row builder wrote
    double stat_t_enqueue = 0, stat_t_wait = 0, stat_t_build = 0, stat_t_total = 0;   // seconds, host-pointer batches
};

}  // namespace

struct qlnlp_handle_s {
    Problem prob;
    std::vector<DeviceState> devs;     // one per device: a handle from qlnlp_create has one
    bool multi = false;                // from qlnlp_create_multi: the single-device entry points refuse it
    std::vector<std::unique_ptr<qlhost::Worker>> drivers;   // multi: one thread per device runs its host-pointer shard

    // host-pointer path: row plan of the batch pattern, registered output buffers.  The driver threads share both and
    // only read them: the plan is built before a shard is handed to a driver.
    std::unique_ptr<qlhost::RowPlan> plan;
    std::vector<Registration> regs;
    int64_t opt_host_chunk = 512;
    int64_t opt_host_threads = 0;      // 0: each device's share of the process's CPUs
    int64_t opt_pin_threads = 1;
    int64_t opt_x_cache = 1;
    int64_t opt_compressible = 1;      // qlnlp_device_alloc: ask for compressible memory where the device has it
};

namespace {

// ---------------------------------------------------------------------------- host planner
struct ModePattern { int nvar; const unsigned char *vi, *vj; int ncon; const unsigned char *ci, *cj; const double* cv; };
ModePattern mode_pattern(int mode)
{
    if (mode == 1) return {QL_NJ_MODE1, QL_PAT_I_MODE1, QL_PAT_J_MODE1, QL_NJC_MODE1, QL_CPAT_I_MODE1, QL_CPAT_J_MODE1, QL_CPAT_V_MODE1};
    if (mode == 2) return {QL_NJ_MODE2, QL_PAT_I_MODE2, QL_PAT_J_MODE2, QL_NJC_MODE2, QL_CPAT_I_MODE2, QL_CPAT_J_MODE2, QL_CPAT_V_MODE2};
    return {QL_NJ_MODE3, QL_PAT_I_MODE3, QL_PAT_J_MODE3, QL_NJC_MODE3, QL_CPAT_I_MODE3, QL_CPAT_J_MODE3, QL_CPAT_V_MODE3};
}
// rows the jump Jacobian keeps (planar_quadruped.jl:262-263)
const int JUMP_KEEP[QL_NX] = {1, 1, 1, 1, 0, 1, 0, 1, 1, 1, 0, 0, 0, 0, 0};

// The block plan of a class: every SPARSE_BLOCK value in value order, with its row and column (the closed-form
// layout), its constant (everything jac_c! assigns that does not depend on Z; 0 elsewhere) and whether it is in the
// VALS stream (layout.h: ql_vals_run_off; the kernel's writer is ql_vals_write_run in true_run.h).  SPARSE_TRUE is the
// sub-sequence of values that are not structural zeros: a non-zero constant, or value-dependent.
int block_plan(const QlClass& c, std::vector<BlockEntry>& plan)
{
    plan.assign((size_t)c.nnz, BlockEntry{});
    int64_t n = 0;
    for (int k = 1; k <= c.N; ++k) {
        const int ncol = (k < c.N) ? QL_NZK : QL_NX;
        for (int j = 0; j < ncol; ++j) {
            const int col = QL_NZK * (k - 1) + j + 1;
            auto put = [&](int row0) { plan[(size_t)n].row = row0 + 1; plan[(size_t)n].col = col; ++n; };
            if (j < QL_NX) {
                if (k == 1) for (int i = 0; i < QL_NX; ++i) put(i);                              // init rows
                if (k == c.N) for (int i = 0; i < QL_NX - 1; ++i) put(c.c_term + i);             // term rows
                if (k >= 2) for (int i = 0; i < QL_NX; ++i) put(c.c_dyn + QL_NX * (k - 2) + i);  // -I block
                if (k < c.N) for (int i = 0; i < QL_NX; ++i) put(c.c_dyn + QL_NX * (k - 1) + i); // RK4 block
                const int jf = (c.init_mode == 1) ? 4 : 6, jo = (c.init_mode == 1) ? 6 : 4;
                if (j == jf) put(c.c_cfirst + (k - 1));
                if (j == jo && k >= c.k_trans) put(c.c_cother + (k - c.k_trans));
                if (j == 1 || j == 2) put(c.c_body + (k - 1));
            } else {
                for (int i = 0; i < QL_NX; ++i) put(c.c_dyn + QL_NX * (k - 1) + i);
                if (k == c.N - 1 && (j == 16 || j == 18)) put(c.c_fctrl);
            }
        }
    }
    std::vector<double> image((size_t)c.nnz, 0.0);
    std::vector<int32_t> vals_pos;             // in VALS order
    vals_pos.reserve((size_t)c.nnz_vals);
    for (int k = 1; k <= c.N; ++k) {
        const int base = ql_run_off(c, k);
        ql_write_run_constants(c, k, image.data() + base);
        const int theta = base + ql_theta_pos(c, k);
        if (k == c.N) { vals_pos.push_back(theta); continue; }
        const bool jump = (k == c.k_trans - 1);
        const ModePattern mp = mode_pattern(k >= c.k_trans ? 3 : c.init_mode);
        for (int e = 0; e < mp.ncon; ++e)
            image[(size_t)(base + ql_rk4_pos(c, k, mp.ci[e], mp.cj[e]))] = (jump && !JUMP_KEEP[mp.ci[e]]) ? 0.0 : mp.cv[e];
        bool theta_done = false;
        for (int e = 0; e < mp.nvar; ++e) {
            if (jump && !JUMP_KEEP[mp.vi[e]]) continue;          // constant zero at the jump knot: stays in the image
            if (mp.vj[e] >= 3 && !theta_done) { vals_pos.push_back(theta); theta_done = true; }
            vals_pos.push_back(base + ql_rk4_pos(c, k, mp.vi[e], mp.vj[e]));
        }
        if (!theta_done) vals_pos.push_back(theta);
    }
    // the VALS stream is the value-dependent entries in value order: a mark per entry says all of it
    if ((int)vals_pos.size() != c.nnz_vals) return fail(QLNLP_ECUDA, "internal: VALS map has %zu entries, layout says %d", vals_pos.size(), c.nnz_vals);
    for (size_t i = 1; i < vals_pos.size(); ++i)
        if (vals_pos[i] <= vals_pos[i - 1]) return fail(QLNLP_ECUDA, "internal: VALS map is not ascending at %zu", i);
    for (int32_t q : vals_pos) plan[(size_t)q].vals = true;
    int nnz_true = 0;
    for (size_t i = 0; i < plan.size(); ++i) {
        plan[i].konst = image[i];
        nnz_true += plan[i].konst != 0.0 || plan[i].vals;
    }
    if (nnz_true != c.nnz_true) return fail(QLNLP_ECUDA, "internal: SPARSE_TRUE has %d entries, layout says %d", nnz_true, c.nnz_true);
    return QLNLP_OK;
}

// Segment plan: per pass, consecutive knots paired.  Two segments share a template id exactly when their staging
// buffers hold the same image once the owner lanes have patched it: the same parity of `start` (the image's offset in
// the buffer), the same knot count, and the same constants and value-dependent positions over [start, end).
void plan_segments(const QlClass& c, const std::vector<BlockEntry>& block, std::vector<QlSeg>& segs, std::vector<int>& seg_begin)
{
    std::map<std::tuple<int, int, std::vector<std::pair<double, bool>>>, int> ids;
    segs.clear();
    seg_begin.assign(1, 0);
    for (int p = 0; p < c.npass; ++p) {
        const int ka = p * QL_LANES + 1, kb = std::min(c.N, ka + QL_LANES - 1);
        for (int k = ka; k <= kb; k += 2) {
            QlSeg s;
            std::memset(&s, 0, sizeof s);
            const int nk = (k + 1 <= kb) ? 2 : 1;
            s.k0 = (short)k;
            s.nk = (signed char)nk;
            s.start = ql_run_off(c, k);
            s.end = (k + nk > c.N) ? c.nnz : ql_run_off(c, k + nk);
            std::vector<std::pair<double, bool>> image;
            for (int i = s.start; i < s.end; ++i) image.emplace_back(block[(size_t)i].konst, block[(size_t)i].vals);
            s.tmpl = (short)ids.emplace(std::make_tuple(s.start & 1, nk, std::move(image)), (int)ids.size()).first->second;
            s.buf = 0;      // unused: the kernel alternates the staging buffers with a running counter (ql_seg_buffer)
            segs.push_back(s);
        }
        seg_begin.push_back((int)segs.size());
    }
}

// ---- what the launcher knows about a kernel ----------------------------------------------------------------------
// The launch policies, each measured on the B200.  One CTA is one warp.
struct KernelSpec {
    const void* fn;
    size_t smem;        // dynamic shared memory per CTA at the problem's N
    int warp_cap;       // most resident CTAs per SM (0: as many as fit)
    bool carveout;      // the library sets the kernel's carve-out to what its resident CTAs need (else: driver default)
    bool pad;           // launched with padded shared memory, so that one CTA more than asked for never fits
    bool pdl;           // programmatic dependent launch
};

// eval_kernel<JM, FASTDIV, RAGGED>; RAGGED: rows addressed through offset tables (qlnlp_eval_ragged_device) instead of
// leading dimensions.  JM_VALS serves the host-pointer path only and is never ragged.
#define QL_EVAL_FNS(JM) {{(const void*)ql::eval_kernel<JM, false, false>, (const void*)ql::eval_kernel<JM, false, true>}, \
                         {(const void*)ql::eval_kernel<JM, true, false>, (const void*)ql::eval_kernel<JM, true, true>}}
const void* const EVAL_FN[NJM][2][2] = {
    QL_EVAL_FNS(ql::JM_NONE), QL_EVAL_FNS(ql::JM_BLOCK), QL_EVAL_FNS(ql::JM_TRUE),
    {{(const void*)ql::eval_kernel<ql::JM_VALS, false, false>, nullptr}, {(const void*)ql::eval_kernel<ql::JM_VALS, true, false>, nullptr}},
};
#undef QL_EVAL_FNS

KernelSpec eval_spec(int N, int jm, bool fast, bool ragged)
{
    // SPARSE_BLOCK: all 8 CTAs per SM that fit (launch() narrows that to 7 for short batches), with padded shared
    // memory.  Since the outputs live in compressible memory the stream no longer waits on DRAM but on the warps' own
    // arithmetic, and more resident warps hide it (profiles/r05_occupancy_sweep.log; the 5-6 warps of
    // profiles/r01_ablation.md section 7 were measured against plain memory).  The other value streams run as many
    // warps as the kernel was compiled for (its __launch_bounds__).
    const bool block = jm == ql::JM_BLOCK;
    const int cap = block ? 8 : jm == ql::JM_NONE ? QL_NONE_WARPS : QL_TRUE_WARPS;
    return {EVAL_FN[jm][fast][ragged], ql::smem_bytes(N, jm), cap, true, block, true};
}

KernelSpec prod_spec(const Problem& p)
{
    const void* fn = p.fastdiv ? (const void*)ql::eval_prod_kernel<true> : (const void*)ql::eval_prod_kernel<false>;
    return {fn, ql::smem_bytes(p.cls.N, ql::JM_PROD), QL_TRUE_WARPS, true, false, true};
}

// the Hessian kernels have not been measured with programmatic dependent launch
KernelSpec hess_spec(const Problem& p, bool prod)
{
    const void* fn = prod ? (p.fastdiv ? (const void*)ql::hess_prod_kernel<true> : (const void*)ql::hess_prod_kernel<false>)
                          : (p.fastdiv ? (const void*)ql::hess_kernel<true> : (const void*)ql::hess_kernel<false>);
    return {fn, ql::hess_smem_bytes(p.cls.N), 0, true, false, false};
}

// static shared memory only; its carve-out has not been measured, so the driver's default stays
KernelSpec kkt_spec() { return {(const void*)ql::kkt_kernel, 0, 0, false, false, true}; }
KernelSpec kkt_factor_spec() { return {(const void*)ql::kkt_factor_kernel, 0, 0, false, false, true}; }
KernelSpec kkt_solve_factored_spec() { return {(const void*)ql::kkt_solve_factored_kernel, 0, 0, false, false, true}; }
KernelSpec kkt_residual_spec() { return {(const void*)ql::kkt_residual_kernel, 0, 0, false, false, true}; }

// the sparse pattern batched evaluations of this problem produce (DENSE handles batch in SPARSE_BLOCK)
int batch_jm(const Problem& p) { return p.jac_mode == QLNLP_JAC_SPARSE_TRUE ? ql::JM_TRUE : ql::JM_BLOCK; }
int std_nnz(const Problem& p) { return p.jac_mode == QLNLP_JAC_SPARSE_TRUE ? p.cls.nnz_true : p.cls.nnz; }
// what the caller sees: the kinematic rows add 8 entries per knot to either pattern and 2 rows per knot to g
int batch_nnz(const Problem& p) { return std_nnz(p) + (p.kin ? 8 * p.cls.N : 0); }
int m_rows(const Problem& p) { return p.cls.m_nlp + (p.kin ? 2 * p.cls.N : 0); }

// One value of the Jacobian row a batched evaluation of the handle returns
struct BatchEntry {
    BlockEntry v;      // a kinematic entry: a constant 0 outside the VALS stream (its rows never take the VALS route)
    int32_t src;       // position in the kernel's row (SPARSE_BLOCK or SPARSE_TRUE order), or -(8 (k-1) + e + 1) for
                       // the kinematic entry e of knot k (qlnlp_kin.cuh)
};

// The Jacobian pattern the caller of the handle sees, in value order: the block plan (DENSE handles batch in
// SPARSE_BLOCK) or its SPARSE_TRUE sub-sequence, with the kinematic rows' 8 entries per knot merged in column-major.
std::vector<BatchEntry> batch_pattern(const Problem& p)
{
    const QlClass& c = p.cls;
    std::vector<BatchEntry> out;
    out.reserve((size_t)batch_nnz(p));
    for (const BlockEntry& e : p.block)
        if (batch_jm(p) == ql::JM_BLOCK || e.konst != 0.0 || e.vals) out.push_back({e, (int32_t)out.size()});
    if (p.kin) {
        static const int COL[8] = {0, 1, 3, 4, 0, 1, 5, 6};
        for (int k = 1; k <= c.N; ++k)
            for (int e = 0; e < 8; ++e)
                out.push_back({{c.m_nlp + 2 * (k - 1) + (e >> 2) + 1, QL_NZK * (k - 1) + COL[e] + 1, 0.0, false}, -(8 * (k - 1) + e + 1)});
        std::sort(out.begin(), out.end(), [](const BatchEntry& a, const BatchEntry& b) {
            return a.v.col != b.v.col ? a.v.col < b.v.col : a.v.row < b.v.row;
        });
    }
    return out;
}

// The constant image and the VALS positions of a row of the handle's batch pattern
void batch_image_and_vals_map(const Problem& p, std::vector<double>& image, std::vector<int32_t>& pos)
{
    const std::vector<BatchEntry> pat = batch_pattern(p);
    image.resize(pat.size());
    pos.clear();
    for (size_t i = 0; i < pat.size(); ++i) {
        image[i] = pat[i].v.konst;
        if (pat[i].v.vals) pos.push_back((int32_t)i);
    }
}

// Row plan of the handle's batch pattern.
int ensure_plan(qlnlp_handle h)
{
    if (h->plan) return QLNLP_OK;
    std::vector<double> image;
    std::vector<int32_t> pos;
    batch_image_and_vals_map(h->prob, image, pos);
    h->plan.reset(new (std::nothrow) qlhost::RowPlan((int64_t)image.size(), image.data(), (int64_t)pos.size(), pos.data()));
    if (!h->plan) return fail(QLNLP_ENOMEM, "out of host memory");
    return QLNLP_OK;
}

int env_int(const char* name, int dflt)
{
    if (const char* e = std::getenv(name)) {
        const int n = std::atoi(e);
        if (n > 0) return n;
    }
    return dflt;
}

// The worker pool of device i of the handle: its share of the CPUs the process may use.  With one process per GPU
// (torchrun) the ranks of a node split the cores (LOCAL_RANK of LOCAL_WORLD_SIZE); a multi-device handle splits its
// share again between its devices; on a multi-socket host the share is taken from the CPUs next to the GPU.
int ensure_pool(qlnlp_handle h, int i)
{
    DeviceState& ds = h->devs[(size_t)i];
    if (ds.pool) return QLNLP_OK;
    const int lws = env_int("LOCAL_WORLD_SIZE", 1);
    const int lr = std::getenv("LOCAL_RANK") ? std::atoi(std::getenv("LOCAL_RANK")) : 0;
    const std::vector<int> all = qlhost::affinity_cpus();
    std::vector<int> near = qlhost::cpus_near_pci_device(ds.pci_bus_id.c_str());
    const int ndev = (int)h->devs.size(), nparts = lws * ndev, part = lr * ndev + i;
    std::vector<int> mine;
    if (near.size() == all.size() || near.empty()) {
        mine = qlhost::cpu_slice(all, part, nparts);
    } else {
        // several CPU groups (sockets): the parts are spread evenly over them
        const int groups = std::max<int>(1, (int)((all.size() + near.size() / 2) / near.size()));
        const int per_group = (nparts + groups - 1) / groups;
        mine = qlhost::cpu_slice(near, part % per_group, per_group);
    }
    int T = (int)mine.size();
    if (h->opt_host_threads > 0) T = (int)h->opt_host_threads;
    T = env_int("QLNLP_HOST_THREADS", T);
    T = std::max(1, std::min(T, 256));
    ds.pool.reset(new (std::nothrow) qlhost::Pool(T, mine, h->opt_pin_threads != 0));
    if (!ds.pool) return fail(QLNLP_ENOMEM, "out of host memory");
    return QLNLP_OK;
}

// Dynamic shared memory to ask for so that `per_sm` CTAs fit on an SM but `per_sm + 1` never do, whatever carve-out the
// kernel runs on (see launch(): programmatic dependent launch and spare CTA slots).
size_t padded_smem(size_t smem_per_sm, size_t smem_optin, int per_sm, size_t smem)
{
    const size_t pad = (smem_per_sm / (size_t)(per_sm + 1) - 1024 + 128) & ~(size_t)127;
    if (pad > smem && (size_t)per_sm * (pad + 1024) <= smem_per_sm && pad <= smem_optin) return pad;
    return smem;
}

// cudaFuncAttributePreferredSharedMemoryCarveout value for `need` bytes of shared memory per SM (see set_carveout)
int carveout_pct(size_t need, size_t smem_per_sm)
{
    static const size_t kCarveKB[] = {0, 8, 16, 32, 64, 100, 132, 164, 196, 228};
    const size_t unified = (smem_per_sm + 65535) / 65536 * 65536;      // 228 KB -> 256 KB
    size_t cfg = smem_per_sm;
    for (size_t kb : kCarveKB)
        if (kb * 1024 >= need) { cfg = std::min(cfg, kb * 1024); break; }
    return (int)std::min<size_t>(100, cfg * 100 / std::max<size_t>(1, unified));
}

int set_carveout(const void* fn, int resident_blocks, size_t smem_per_block, size_t smem_per_sm)
{
    static std::map<const void*, size_t> g_need;
    static std::mutex g_mu;                    // the devices of a multi-device handle are set up from their driver threads
    std::lock_guard<std::mutex> lk(g_mu);
    size_t& need = g_need[fn];
    need = std::max(need, (size_t)resident_blocks * (smem_per_block + 1024));
    // The attribute is a percentage of the SM's UNIFIED L1 + shared memory (256 KB on sm_100; measured: 50 -> 132 KB,
    // 58..65 -> 164 KB, 72 -> 196 KB, >= 79 -> 228 KB), rounded up to a carve-out the SM supports (0, 8, 16, 32, 64, 100,
    // 132, 164, 196, 228 KB).  Ask for the smallest of those that holds `need`.  (Taking the percentage of the 228 KB
    // shared-memory maximum instead left the kernel without a Jacobian on 228 KB of shared memory and 28 KB of L1:
    // ncu launch__shared_mem_config_size; 46 % of its cost-table loads missed L1.  profiles/r02_kernel_ab.md)
    CUDA_TRY(cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, carveout_pct(need, smem_per_sm)));
    return QLNLP_OK;
}

// Launch geometry of kernel `k` on the device `ds`: the resident CTAs per SM, and the L1 carve-out they leave.  Cached
// per device on the first call.
int kernel_geometry(DeviceState& ds, const KernelSpec& k, int* blocks_per_sm)
{
    const auto key = std::make_pair(k.fn, k.smem);
    auto it = ds.blocks_per_sm.find(key);
    if (it != ds.blocks_per_sm.end()) { *blocks_per_sm = it->second; return QLNLP_OK; }
    if (k.smem > ds.smem_optin) return fail(QLNLP_EINVAL, "the kernel needs %zu B of shared memory per warp (> %zu)", k.smem, ds.smem_optin);
    if (k.carveout) {
        // the attributes are per FUNCTION, shared by every handle of the process: always raise the limit to the
        // device's, never to this handle's own (possibly smaller) requirement
        CUDA_TRY(cudaFuncSetAttribute(k.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ds.smem_optin));
        CUDA_TRY(cudaFuncSetAttribute(k.fn, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    }
    int nb = 0;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k.fn, QL_LANES, k.smem));
    if (nb < 1) return fail(QLNLP_ECUDA, "kernel does not fit on an SM");
    if (k.warp_cap) nb = std::min(nb, k.warp_cap);
    if (k.carveout) {
        // Shared memory the resident warps really need: whatever the SM has beyond that serves as L1 (the cost table
        // and the boundary states are re-read by every warp).  The attribute belongs to the FUNCTION, so it only ever
        // grows (handles of other horizons share it).
        const size_t per_block = k.pad ? padded_smem(ds.smem_per_sm, ds.smem_optin, nb, k.smem) : k.smem;
        if (int rc = set_carveout(k.fn, nb, per_block, ds.smem_per_sm)) return rc;
    }
    ds.blocks_per_sm.emplace(key, nb);
    *blocks_per_sm = nb;
    return QLNLP_OK;
}

int check_handle(qlnlp_handle h)
{
    if (!h) return fail(QLNLP_EINVAL, "null handle");
    return QLNLP_OK;
}

// Whether work on `stream` is being captured into a graph (the legacy default stream never is)
bool capturing(cudaStream_t stream)
{
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    return stream && cudaStreamIsCapturing(stream, &cap) == cudaSuccess && cap != cudaStreamCaptureStatusNone;
}

// First-use set-up (allocations, blocking copies, a device synchronise) would invalidate a graph capture: the call
// that needs it is refused before it makes any such call, and the caller's capture goes on.
int refuse_setup_in_capture(cudaStream_t stream, const char* what)
{
    if (!capturing(stream)) return QLNLP_OK;
    return fail(QLNLP_EINVAL, "%s: first use inside a CUDA-graph capture, which cannot allocate or synchronise; warm the "
                "handle with one such call outside the capture before capturing", what);
}

// Binds one device of a handle (first call: tables, occupancy, streams), all or nothing: a failed set-up releases what
// it made (`state` is replaced once the set-up is complete).  The caller holds a DeviceGuard.  `stream`: the stream the
// call launches on (set-up is refused while it is being captured).
int ensure_device(const Problem& p, DeviceState& state, cudaStream_t stream = nullptr)
{
    if (state.ready) return QLNLP_OK;
    if (int rc = refuse_setup_in_capture(stream, "set-up of the handle")) return rc;
    DeviceState ds{state.device};
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(QLNLP_ENODEVICE, "no CUDA device available (%s); this library has no CPU path",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (ds.device < 0 || ds.device >= ndev) return fail(QLNLP_EINVAL, "device %d out of range (0..%d)", ds.device, ndev - 1);
    CUDA_TRY(cudaSetDevice(ds.device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, ds.device));
    if (prop.major != 10)
        return fail(QLNLP_ENODEVICE, "device %d is sm_%d%d; this build targets sm_100a (B200) only", ds.device, prop.major,
                    prop.minor);
    ds.sm_count = prop.multiProcessorCount;
    ds.smem_per_sm = prop.sharedMemPerMultiprocessor;
    ds.smem_optin = prop.sharedMemPerBlockOptin;
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, ds.device) == cudaSuccess) ds.pci_bus_id = bus;

    if (int rc = upload(ds.d_cost, p.cost.data(), p.cost.size(), false)) return rc;
    if (int rc = upload(ds.d_x0xf, p.x0xf, 2 * QL_NX, false)) return rc;
    if (int rc = upload(ds.d_segs, p.segs.data(), p.segs.size(), false)) return rc;
    if (int rc = upload(ds.d_seg_begin, p.seg_begin.data(), p.seg_begin.size(), false)) return rc;

    // the eval kernels' attributes are set here, at the first evaluation, whatever the handle launches later
    for (int wj = 0; wj < NJM; ++wj)
        for (int rg = 0; rg < (wj == ql::JM_VALS ? 1 : 2); ++rg) {
            int nb = 0;
            if (int rc = kernel_geometry(ds, eval_spec(p.cls.N, wj, p.fastdiv, rg != 0), &nb)) return rc;
        }
    cudaStream_t s = nullptr;
    cudaEvent_t ev = nullptr;
    for (auto& ln : ds.lanes) {
        CUDA_TRY(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
        ln.stream.reset(s);
        CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        ln.done.reset(ev);
    }
    CUDA_TRY(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    ds.one.stream.reset(s);
    if (int rc = device_alloc(ds.ticket_pool, 32 * (TICKET_POOL + GRAPH_TICKETS))) return rc;
    CUDA_TRY(cudaMemset(ds.ticket_pool.get(), 0, 128 * (TICKET_POOL + GRAPH_TICKETS)));
    ds.graph_tickets = std::make_shared<GraphTickets>();
    for (int i = TICKET_POOL + GRAPH_TICKETS - 1; i >= TICKET_POOL; --i) ds.graph_tickets->free.push_back(i);
    CUDA_TRY(cudaDeviceSynchronize());         // the set-up copies (upload)
    ds.ready = true;
    ds.pool = std::move(state.pool);           // row builders started before the set-up (qlnlp_host_output_register)
    state = std::move(ds);
    return QLNLP_OK;
}

// Work counter of a stream (launches on one stream are ordered, so they can share it; the kernel's last CTA re-arms
// it).  Concurrent launches on the device on different streams get different counters.
int stream_ticket(DeviceState& ds, cudaStream_t stream, unsigned** out)
{
    auto it = ds.tickets.find(stream);
    if (it == ds.tickets.end()) {
        if (ds.ticket_pool_used >= TICKET_POOL) {
            // Every counter of the pre-zeroed pool belongs to a stream.  Streams come and go (torch pools), so wait
            // for the handle's outstanding launches and start the pool over rather than allocating (an allocation
            // here would make the launch illegal inside a CUDA-graph capture, and a faulted kernel could leave a
            // counter un-re-armed: the reset also heals that).
            cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
            cudaStreamIsCapturing(stream, &cap);
            if (cap != cudaStreamCaptureStatusNone)
                return fail(QLNLP_EINVAL, "more than %d streams used with this handle: cannot recycle work counters during a graph capture", TICKET_POOL);
            CUDA_TRY(cudaDeviceSynchronize());
            CUDA_TRY(cudaMemset(ds.ticket_pool.get(), 0, 128 * TICKET_POOL));
            CUDA_TRY(cudaDeviceSynchronize());
            ds.tickets.clear();
            ds.ticket_pool_used = 0;
        }
        unsigned* d = ds.ticket_pool.get() + 32 * ds.ticket_pool_used++;      // zeroed (and synchronised) at set-up
        it = ds.tickets.emplace(stream, d).first;
    }
    *out = it->second;
    return QLNLP_OK;
}

// Work counter of a launch on `stream`.  An eager launch takes the stream's counter.  A launch captured into a graph
// takes a counter its graph owns (GraphTickets), never a stream's: a replay may run on any stream, beside eager work
// on the capture stream and beside replays of other graphs captured there, and each grid needs a counter no other
// running grid draws from.  Launches of one capture sequence on one stream are ordered, so they share one.
int launch_ticket(DeviceState& ds, cudaStream_t stream, unsigned** out)
{
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    unsigned long long id = 0;
    cudaGraph_t graph = nullptr;
    if (cudaStreamGetCaptureInfo(stream, &cap, &id, &graph) != cudaSuccess || cap != cudaStreamCaptureStatusActive)
        return stream_ticket(ds, stream, out);
    GraphTickets& gt = *ds.graph_tickets;
    const auto key = std::make_pair(id, stream);
    int index = -1;
    {
        std::lock_guard<std::mutex> lk(gt.mu);
        auto it = gt.live.find(key);
        if (it != gt.live.end()) {
            *out = ds.ticket_pool.get() + 32 * it->second;
            return QLNLP_OK;
        }
        if (gt.free.empty())
            return fail(QLNLP_EINVAL, "%d captured graphs of this handle hold work counters: destroy some before capturing more",
                        GRAPH_TICKETS);
        index = gt.free.back();
        gt.free.pop_back();
        gt.live.emplace(key, index);
    }
    // the graph takes the only reference; the CUDA calls run outside the lock (a release may run the destructor)
    GraphTicket* t = new (std::nothrow) GraphTicket{ds.graph_tickets, key, index};
    if (!t) {
        std::lock_guard<std::mutex> lk(gt.mu);
        gt.live.erase(key);
        gt.free.push_back(index);
        return fail(QLNLP_ENOMEM, "out of host memory");
    }
    cudaUserObject_t obj = nullptr;
    if (cudaError_t e = cudaUserObjectCreate(&obj, t, release_graph_ticket, 1, cudaUserObjectNoDestructorSync)) {
        release_graph_ticket(t);
        return fail(QLNLP_ECUDA, "cudaUserObjectCreate: %s", cudaGetErrorString(e));
    }
    if (cudaError_t e = cudaGraphRetainUserObject(graph, obj, 1, cudaGraphUserObjectMove)) {
        cudaUserObjectRelease(obj, 1);
        return fail(QLNLP_ECUDA, "cudaGraphRetainUserObject: %s", cudaGetErrorString(e));
    }
    *out = ds.ticket_pool.get() + 32 * index;
    return QLNLP_OK;
}

// The one launch of every kernel that hands out work with a ticket: B evaluations of record `P` on `stream`, on at most
// `cap` resident CTAs per SM.  `info`: the launch_info record to fill (eval launches).
template <typename R>
int launch_kernel(DeviceState& ds, const KernelSpec& k, int64_t B, R& P, cudaStream_t stream, int cap = INT_MAX,
                  int64_t* info = nullptr)
{
    int per_sm = 0;
    if (int rc = kernel_geometry(ds, k, &per_sm)) return rc;
    per_sm = std::min(per_sm, cap);
    const int grid = (int)std::min<int64_t>(B, (int64_t)ds.sm_count * per_sm);
    if (int rc = launch_ticket(ds, stream, &P.ticket)) return rc;
    // With programmatic dependent launch the next grid's CTAs are placed as soon as an SM has room for one.  The
    // SPARSE_BLOCK kernel can run on fewer CTAs per SM than would fit (7 of 8 for short batches): a spare slot
    // would take a CTA of the next grid while this grid is still running at full strength, and the next grid would
    // start out unevenly spread over the SMs (measured: -5 % on the headline once another handle had raised the
    // kernel's carve-out to 228 KB).  Ask for enough shared memory per CTA that per_sm + 1 of them never fit.
    // (Only that kernel: the others are capped by their registers, and padding them would cost L1.)
    const size_t smem = k.pad ? padded_smem(ds.smem_per_sm, ds.smem_optin, per_sm, k.smem) : k.smem;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(QL_LANES);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    // programmatic dependent launch: back-to-back launches on a stream overlap the next grid's start-up with this
    // grid's drain (B = 4,096: +1 % full evaluation, +4..6 % for the compact-output kernels; the kernels wait for their
    // predecessors before they touch any data, see griddepcontrol.wait in eval_kernel)
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = k.pdl ? 1 : 0;
    void* args[] = {&P};
    CUDA_TRY(cudaLaunchKernelExC(&cfg, k.fn, args));
    if (info) {
        info[0] = grid;
        info[1] = QL_LANES;
        info[2] = (int64_t)smem;
        info[3] = per_sm;
        info[4] = ds.sm_count;
    }
    return QLNLP_OK;
}

// The problem fields the launch records share
template <typename R>
void set_problem(R& P, const Problem& p, const DeviceState& ds)
{
    P.c = p.cls;
    P.rmb = p.rmb; P.rmf = p.rmf; P.rIb = p.rIb;
    P.cost = ds.d_cost.get();
    P.npad = p.npad;
    if constexpr (std::is_base_of<ql::Launch, R>::value) {
        P.x0_def = ds.d_x0xf.get();
        P.xf_def = ds.d_x0xf.get() + QL_NX;
    }
}

// Device scratch of at least n doubles for eager work on one stream, grown only.  (A launch captured into a graph
// takes scratch its graph owns instead: launch_scratch.)
int grow_scratch(Scratch& sc, size_t n, double** out)
{
    if (sc.cap < n) {
        if (sc.ptr) CUDA_TRY(cudaDeviceSynchronize());      // earlier launches may still use it
        sc = Scratch();
        if (int rc = device_alloc(sc.ptr, n)) return rc;
        sc.cap = n;
    }
    *out = sc.ptr.get();
    return QLNLP_OK;
}

// Scratch of n doubles for the launches of one call on `stream`.  Eager: the stream's grow-only block in `per_stream`.
// Inside a graph capture: a block of the graph's own, allocated here and freed by end_scratch after the call's last
// kernel (graph memory nodes).  A replay then shares no scratch with eager work or with other graphs, and no eager
// call can free a block a graph still points to.
int launch_scratch(std::map<cudaStream_t, Scratch>& per_stream, cudaStream_t stream, size_t n, double** out, bool* owned)
{
    *owned = capturing(stream);
    if (*owned) {
        CUDA_TRY(cudaMallocAsync(reinterpret_cast<void**>(out), sizeof(double) * n, stream));
        return QLNLP_OK;
    }
    return grow_scratch(per_stream[stream], n, out);
}

int end_scratch(double* ptr, bool owned, cudaStream_t stream)
{
    if (owned) CUDA_TRY(cudaFreeAsync(ptr, stream));
    return QLNLP_OK;
}

// End of a call that reads or writes caller-owned host memory: wait for `stream` whatever happened (copies may still be
// in flight), and report the first error.
int finish(cudaStream_t stream, int rc, const char* what)
{
    const std::string msg = g_err;
    const cudaError_t e = cudaStreamSynchronize(stream);
    if (rc == QLNLP_OK && e != cudaSuccess) return fail(QLNLP_ECUDA, "%s: %s", what, cudaGetErrorString(e));
    g_err = msg;
    return rc;
}

// Argument checks of a batch on device pointers (rg: a ragged batch) or, with `host`, on host pointers: host logic
// only, before any device is touched.  The kernels read Z themselves; on host pointers the row builder writes jac.
int check_batch(const Problem& p, int64_t B, const qlnlp_batch_io* io, const qlnlp_ragged_io* rg, bool host = false)
{
    const QlClass& c = p.cls;
    if (B < 0) return fail(QLNLP_EINVAL, "negative batch");
    if (!io || !io->Z) return fail(QLNLP_EINVAL, "io->Z is required");
    if (rg) {
        if (!rg->z_off || (io->g && !rg->g_off) || (io->jac && !rg->jac_off))
            return fail(QLNLP_EINVAL, "ragged launch: offset tables are required for every requested array");
    } else {
        if (io->ldz < c.n_nlp) return fail(QLNLP_EINVAL, "ldz %lld < n_nlp %d", (long long)io->ldz, c.n_nlp);
        if (io->grad && io->ldgrad < c.n_nlp) return fail(QLNLP_EINVAL, "ldgrad %lld < n_nlp %d", (long long)io->ldgrad, c.n_nlp);
        if (io->g && io->ldg < m_rows(p)) return fail(QLNLP_EINVAL, "ldg %lld < m_nlp %d", (long long)io->ldg, m_rows(p));
        if (io->jac && io->ldjac < batch_nnz(p)) return fail(QLNLP_EINVAL, "ldjac %lld < nnz %d", (long long)io->ldjac, batch_nnz(p));
    }
    if (!host && (reinterpret_cast<uintptr_t>(io->Z) & 7) != 0) return fail(QLNLP_EINVAL, "Z must be 8-byte aligned");
    if (host && io->jac && (reinterpret_cast<uintptr_t>(io->jac) & 7) != 0) return fail(QLNLP_EINVAL, "jac must be 8-byte aligned");
    return QLNLP_OK;
}

// One launch of the evaluator over arguments that have passed check_batch (B > 0).  jm_force: the value stream to
// write instead of the batch pattern's (JM_VALS for the host-pointer paths).
int launch(const Problem& p, DeviceState& ds, int64_t B, const qlnlp_batch_io* io, cudaStream_t stream, int jm_force = -1,
           const qlnlp_ragged_io* rg = nullptr, const RagTable* table = nullptr, const int32_t* class_of = nullptr)
{
    ql::Launch P;
    set_problem(P, p, ds);
    if (rg) P.c = table->layout;
    P.classes = rg ? reinterpret_cast<const ql::QlRagClass*>(table->d_classes.get()) : nullptr;
    P.cls_of = rg ? reinterpret_cast<const int*>(class_of) : nullptr;
    P.nseg = (int)p.segs.size();
    P.segs = ds.d_segs.get();
    P.seg_begin = ds.d_seg_begin.get();
    P.io = *io;
    P.B = B;
    P.index = rg ? reinterpret_cast<const long long*>(rg->index) : nullptr;
    P.z_off = rg ? reinterpret_cast<const long long*>(rg->z_off) : nullptr;
    P.g_off = rg ? reinterpret_cast<const long long*>(rg->g_off) : nullptr;
    P.j_off = rg ? reinterpret_cast<const long long*>(rg->jac_off) : nullptr;
    P.bulk = (io->jac && (reinterpret_cast<uintptr_t>(io->jac) & 15) == 0 && (rg || (io->ldjac & 1) == 0)) ? 1 : 0;
    if (rg) P.zbulk = ((reinterpret_cast<uintptr_t>(io->Z) & 15) == 0 && (rg->flags & QLNLP_RAGGED_Z_PADDED)) ? 1 : 0;
    else P.zbulk = ((reinterpret_cast<uintptr_t>(io->Z) & 15) == 0 && (io->ldz & 1) == 0) ? 1 : 0;   // ldz even > n_nlp (odd)

    const int wj = io->jac ? (jm_force >= 0 ? jm_force : batch_jm(p)) : ql::JM_NONE;
    int cap = INT_MAX;
    if (!rg && wj != ql::JM_VALS)      // a plain launch runs on no more CTAs per SM than the ragged instantiation
        if (int rc = kernel_geometry(ds, eval_spec(p.cls.N, wj, p.fastdiv, true), &cap)) return rc;
    // SPARSE_BLOCK: 8 CTAs per SM, 7 for short batches (fewer than 8 evaluations per warp).  B = 4,096 at 7 / 8 / the
    // former 6 or 5: full 24.8 / 24.2 / 24.6, g+J 27.8 / 26.9 / 26.0 M evals/s (profiles/r05_occupancy_sweep.log)
    if (wj == ql::JM_BLOCK) cap = std::min(cap, B < 8 * (int64_t)ds.sm_count * 7 ? 7 : 8);
    const KernelSpec k = rg ? eval_spec(table->layout.N, wj, table->fastdiv, true) : eval_spec(p.cls.N, wj, p.fastdiv, false);
    return launch_kernel(ds, k, B, P, stream, cap, ds.last_launch);
}

// The class table of a ragged launch over the single-device handles `hs` (all on one device, already bound to it),
// cached in the device state of hs[0].  A new class set is refused while `stream` is being captured.
int ragged_table(const qlnlp_handle* hs, int ncls, cudaStream_t stream, const RagTable** out)
{
    DeviceState& lead = hs[0]->devs[0];
    std::vector<uint64_t> key((size_t)ncls);
    for (int i = 0; i < ncls; ++i) key[(size_t)i] = hs[i]->prob.serial;
    auto it = lead.rag_tables.find(key);
    if (it != lead.rag_tables.end()) { *out = &it->second; return QLNLP_OK; }
    if (int rc = refuse_setup_in_capture(stream, "ragged launch over a new set of classes")) return rc;
    RagTable t;
    t.fastdiv = true;
    t.layout = hs[0]->prob.cls;
    // device records are QL_RAGCLASS_BYTES apart (the kernel copies whole slots)
    std::vector<unsigned char> packed((size_t)ncls * QL_RAGCLASS_BYTES, 0);
    for (int i = 0; i < ncls; ++i) {
        const Problem& p = hs[i]->prob;
        const DeviceState& ds = hs[i]->devs[0];
        ql::QlRagClass r;
        std::memset(&r, 0, sizeof r);
        r.c = p.cls;
        r.rmb = p.rmb; r.rmf = p.rmf; r.rIb = p.rIb;
        r.cost = ds.d_cost.get();
        r.x0_def = ds.d_x0xf.get();
        r.xf_def = ds.d_x0xf.get() + QL_NX;
        r.segs = ds.d_segs.get();
        r.seg_begin = ds.d_seg_begin.get();
        r.npad = p.npad;
        r.nseg = (int)p.segs.size();
        t.fastdiv = t.fastdiv && p.fastdiv;
        if (p.cls.N > t.layout.N) t.layout = p.cls;
        std::memcpy(packed.data() + (size_t)i * QL_RAGCLASS_BYTES, &r, sizeof r);
    }
    if (int rc = upload(t.d_classes, packed.data(), packed.size())) return rc;
    *out = &lead.rag_tables.emplace(key, std::move(t)).first->second;
    return QLNLP_OK;
}

// ---- opt-in kinematic rows (qlnlp_kin.cuh) ---------------------------------------------------------------------
int ensure_kin(const Problem& p, DeviceState& ds, cudaStream_t stream)
{
    if (ds.d_kin_map) return QLNLP_OK;
    if (int rc = refuse_setup_in_capture(stream, "kinematic rows")) return rc;
    std::vector<int32_t> map;
    for (const BatchEntry& e : batch_pattern(p)) map.push_back(e.src);
    return upload(ds.d_kin_map, map.data(), map.size());
}

// launch() for a problem with kinematic rows: io describes the CALLER's arrays (g rows of m_nlp + 2N, jac rows of
// nnz + 8N).  The fused kernel writes the reference's g rows in place and its Jacobian values into a scratch row per
// evaluation; two small kernels append / interleave the kinematic part.
int launch_kin(const Problem& p, DeviceState& ds, int64_t B, const qlnlp_batch_io* io, cudaStream_t stream)
{
    const QlClass& c = p.cls;
    if (int rc = ensure_kin(p, ds, stream)) return rc;
    qlnlp_batch_io d = *io;
    const int64_t lds = (std_nnz(p) + 1) & ~1;
    bool owned = false;
    if (io->jac) {
        if (int rc = launch_scratch(ds.kin_scratch, stream, (size_t)(B * lds), &d.jac, &owned)) return rc;
        d.ldjac = lds;
    }
    if (int rc = launch(p, ds, B, &d, stream)) return rc;
    const int threads = 256;
    if (io->g) {
        const long long total = (long long)B * 2 * c.N;
        ql::kin_g_kernel<<<(unsigned)((total + threads - 1) / threads), threads, 0, stream>>>(io->Z, io->ldz, io->g, io->ldg, B, c.N, c.m_nlp);
        CUDA_TRY(cudaGetLastError());
    }
    if (io->jac) {
        const int nnz_out = batch_nnz(p);
        const long long total = (long long)B * nnz_out;
        ql::kin_expand_kernel<<<(unsigned)((total + threads - 1) / threads), threads, 0, stream>>>(
            ds.d_kin_map.get(), nnz_out, d.jac, lds, io->Z, io->ldz, io->jac, io->ldjac, B);
        CUDA_TRY(cudaGetLastError());
    }
    return end_scratch(d.jac, owned, stream);
}

// ---- Lagrangian Hessian ----------------------------------------------------------------------------------------
void hessian_structure(const QlClass& c, int64_t* rows, int64_t* cols)
{
    int64_t n = 0;
    for (int k = 1; k <= c.N; ++k) {
        const int64_t base = (int64_t)QL_NZK * (k - 1);
        if (k == c.N) {
            for (int i = 0; i < QL_NX; ++i) { rows[n] = base + i + 1; cols[n] = base + i + 1; ++n; }
            continue;
        }
        const int mode = (k >= c.k_trans) ? 3 : c.init_mode;
        const int len = mode == 3 ? QL_HESS_LEN_MODE3 : QL_HESS_LEN_MODE1;
        const unsigned char* R = mode == 1 ? QL_HESS_R_MODE1 : mode == 2 ? QL_HESS_R_MODE2 : QL_HESS_R_MODE3;
        const unsigned char* C = mode == 1 ? QL_HESS_C_MODE1 : mode == 2 ? QL_HESS_C_MODE2 : QL_HESS_C_MODE3;
        for (int e = 0; e < len; ++e) { rows[n] = base + R[e] + 1; cols[n] = base + C[e] + 1; ++n; }
    }
}

// Argument checks of the Hessian entry points: Z, the multipliers and one output row of `width` values per evaluation.
// Host logic only, before any device is touched.
int check_hessian(const Problem& p, int64_t B, const double* Z, int64_t ldz, const double* lam, int64_t ldlam,
                  const double* out, int64_t ldout, int64_t width)
{
    const QlClass& c = p.cls;
    if (B < 0) return fail(QLNLP_EINVAL, "negative batch");
    if (!Z || !lam || !out) return fail(QLNLP_EINVAL, "Z, lambda and the output are required");
    if (ldz < c.n_nlp || ldlam < c.m_nlp || ldout < width) return fail(QLNLP_EINVAL, "leading dimension too small");
    return QLNLP_OK;
}

template <typename R>
void set_hessian(R& P, const Problem& p, const DeviceState& ds, int64_t B, const double* Z, int64_t ldz,
                 const double* sigma, double sigma0, const double* lam, int64_t ldlam)
{
    set_problem(P, p, ds);
    P.Z = Z; P.ldz = ldz;
    P.lam = lam; P.ldlam = ldlam;
    P.sigma = sigma; P.sigma0 = sigma0;
    P.B = B;
    P.zbulk = ((reinterpret_cast<uintptr_t>(Z) & 15) == 0 && (ldz & 1) == 0) ? 1 : 0;
}

int launch_hessian(const Problem& p, DeviceState& ds, int64_t B, const double* Z, int64_t ldz, const double* sigma,
                   double sigma0, const double* lam, int64_t ldlam, double* H, int64_t ldh, cudaStream_t stream)
{
    ql::HessLaunch P;
    set_hessian(P, p, ds, B, Z, ldz, sigma, sigma0, lam, ldlam);
    P.H = H; P.ldh = ldh;
    P.bulk = ((reinterpret_cast<uintptr_t>(H) & 15) == 0 && (ldh & 1) == 0) ? 1 : 0;
    return launch_kernel(ds, hess_spec(p, false), B, P, stream);
}

// ---- matrix-free products (MOI :JacVec / :HessVec) ---------------------------------------------------------------
int check_products(const Problem& p, int64_t B, const qlnlp_batch_io* io, const qlnlp_product_io* pv)
{
    const QlClass& c = p.cls;
    const int m = m_rows(p);
    if (!pv) return fail(QLNLP_EINVAL, "pv is required");
    if (int rc = check_batch(p, B, io, nullptr)) return rc;
    if (io->jac) return fail(QLNLP_EINVAL, "io->jac must be NULL: the product launch writes no Jacobian values");
    if (!pv->w && !pv->y) return fail(QLNLP_EINVAL, "pv->w or pv->y is required");
    if (!pv->w != !pv->jw) return fail(QLNLP_EINVAL, "pv->jw is required iff pv->w is set");
    if (!pv->y != !pv->jty) return fail(QLNLP_EINVAL, "pv->jty is required iff pv->y is set");
    if (pv->w && (pv->ldw < c.n_nlp || pv->ldjw < m))
        return fail(QLNLP_EINVAL, "ldw %lld < n_nlp %d or ldjw %lld < m_nlp %d", (long long)pv->ldw, c.n_nlp, (long long)pv->ldjw, m);
    if (pv->y && (pv->ldy < m || pv->ldjty < c.n_nlp))
        return fail(QLNLP_EINVAL, "ldy %lld < m_nlp %d or ldjty %lld < n_nlp %d", (long long)pv->ldy, m, (long long)pv->ldjty, c.n_nlp);
    for (const void* a : {(const void*)pv->w, (const void*)pv->jw, (const void*)pv->y, (const void*)pv->jty})
        if ((reinterpret_cast<uintptr_t>(a) & 7) != 0) return fail(QLNLP_EINVAL, "arrays must be 8-byte aligned");
    return QLNLP_OK;
}

// One fused launch of eval_prod_kernel: what launch() does for a plain batch, with J w / J' y in place of a value stream.
int launch_products(const Problem& p, DeviceState& ds, int64_t B, const qlnlp_batch_io* io, const qlnlp_product_io* pv,
                    cudaStream_t stream)
{
    ql::ProdLaunch P;
    std::memset(&P, 0, sizeof P);
    set_problem(P, p, ds);
    P.io = *io;
    P.B = B;
    P.zbulk = ((reinterpret_cast<uintptr_t>(io->Z) & 15) == 0 && (io->ldz & 1) == 0) ? 1 : 0;
    P.pv = *pv;
    P.kin = p.kin ? 1 : 0;
    return launch_kernel(ds, prod_spec(p), B, P, stream);
}

int check_hess_products(const Problem& p, int64_t B, const double* Z, int64_t ldz, const double* lam, int64_t ldlam,
                        const double* V, int64_t ldv, const double* HV, int64_t ldhv)
{
    if (int rc = check_hessian(p, B, Z, ldz, lam, ldlam, HV, ldhv, p.cls.n_nlp)) return rc;
    if (!V) return fail(QLNLP_EINVAL, "V is required");
    if (ldv < p.cls.n_nlp) return fail(QLNLP_EINVAL, "leading dimension too small");
    for (const void* a : {(const void*)Z, (const void*)lam, (const void*)V, (const void*)HV})
        if ((reinterpret_cast<uintptr_t>(a) & 7) != 0) return fail(QLNLP_EINVAL, "arrays must be 8-byte aligned");
    return QLNLP_OK;
}

int launch_hess_products(const Problem& p, DeviceState& ds, int64_t B, const double* Z, int64_t ldz, const double* sigma,
                         double sigma0, const double* lam, int64_t ldlam, const double* V, int64_t ldv, double* HV,
                         int64_t ldhv, cudaStream_t stream)
{
    ql::HessProdLaunch P;
    std::memset(&P, 0, sizeof P);
    set_hessian(P, p, ds, B, Z, ldz, sigma, sigma0, lam, ldlam);
    P.V = V; P.ldv = ldv;
    P.HV = HV; P.ldhv = ldhv;
    return launch_kernel(ds, hess_spec(p, true), B, P, stream);
}

// ---- batched KKT solve (qlnlp_kkt.cuh) --------------------------------------------------------------------------
// Argument checks: host logic only, before any device is touched.
int check_kkt(const Problem& p, int64_t B, const qlnlp_kkt_io* io)
{
    const QlClass& c = p.cls;
    if (B < 0) return fail(QLNLP_EINVAL, "negative batch");
    if (!io || !io->hess || !io->jac || !io->dc || !io->r1 || !io->r2 || !io->px || !io->pl || !io->status)
        return fail(QLNLP_EINVAL, "io, hess, jac, dc, r1, r2, px, pl and status are required");
    const int64_t n = c.n_nlp, m = c.m_nlp;
    if (io->ldhess < ql_hess_nnz(c)) return fail(QLNLP_EINVAL, "ldhess %lld < nnz_hess %d", (long long)io->ldhess, ql_hess_nnz(c));
    if (io->ldjac < c.nnz_true) return fail(QLNLP_EINVAL, "ldjac %lld < nnz %d", (long long)io->ldjac, c.nnz_true);
    if (io->sx && io->ldsx < n) return fail(QLNLP_EINVAL, "ldsx %lld < n_nlp %lld", (long long)io->ldsx, (long long)n);
    if (io->ldr1 < n || io->ldpx < n)
        return fail(QLNLP_EINVAL, "ldr1 %lld / ldpx %lld < n_nlp %lld", (long long)io->ldr1, (long long)io->ldpx, (long long)n);
    if (io->lddc < m || io->ldr2 < m || io->ldpl < m)
        return fail(QLNLP_EINVAL, "lddc %lld / ldr2 %lld / ldpl %lld < m_nlp %lld", (long long)io->lddc, (long long)io->ldr2,
                    (long long)io->ldpl, (long long)m);
    for (const void* a : {(const void*)io->hess, (const void*)io->jac, (const void*)io->sx, (const void*)io->dc,
                          (const void*)io->r1, (const void*)io->r2, (const void*)io->px, (const void*)io->pl})
        if ((reinterpret_cast<uintptr_t>(a) & 7) != 0) return fail(QLNLP_EINVAL, "arrays must be 8-byte aligned");
    if ((reinterpret_cast<uintptr_t>(io->status) & 3) != 0) return fail(QLNLP_EINVAL, "status must be 4-byte aligned");
    return QLNLP_OK;
}

// Per-value tables of the kernel, from the host structures: for every SPARSE_TRUE value its slot in the local Jacobian
// of its knot (ql::kkt_slot_row) and its column inside the knot; then for every Hessian value its row and column inside
// the knot (lower triangle).
int ensure_kkt_tables(const Problem& p, DeviceState& ds, cudaStream_t stream)
{
    if (ds.d_kkt_tab) return QLNLP_OK;
    if (int rc = refuse_setup_in_capture(stream, "KKT solve")) return rc;
    const QlClass& c = p.cls;
    const int nh = ql_hess_nnz(c);
    const std::vector<BatchEntry> jac = batch_pattern(p);       // SPARSE_TRUE: the only pattern the KKT solve takes
    std::vector<unsigned short> tab(jac.size() + nh);
    for (size_t e = 0; e < jac.size(); ++e) {
        const int k = (jac[e].v.col - 1) / QL_NZK + 1, j = (jac[e].v.col - 1) % QL_NZK;
        int s = 0;
        while (s < ql::KKT_SLOTS && ql::kkt_slot_row(c, k, s) != jac[e].v.row - 1) ++s;
        if (s == ql::KKT_SLOTS) return fail(QLNLP_ECUDA, "internal: Jacobian row %d has no slot at knot %d", jac[e].v.row, k);
        tab[e] = (unsigned short)(s | j << 8);
    }
    std::vector<int64_t> rows(nh), cols(nh);
    hessian_structure(c, rows.data(), cols.data());
    for (int e = 0; e < nh; ++e) {
        const int r = (int)((rows[e] - 1) % QL_NZK), q = (int)((cols[e] - 1) % QL_NZK);
        tab[jac.size() + e] = (unsigned short)(std::max(r, q) | std::min(r, q) << 8);
    }
    return upload(ds.d_kkt_tab, tab.data(), tab.size());
}

int launch_kkt(const Problem& p, DeviceState& ds, int64_t B, const qlnlp_kkt_io* io, cudaStream_t stream)
{
    const QlClass& c = p.cls;
    if (int rc = ensure_kkt_tables(p, ds, stream)) return rc;
    const KernelSpec k = kkt_spec();
    int per_sm = 0;
    if (int rc = kernel_geometry(ds, k, &per_sm)) return rc;
    // the scratch holds one factor per resident warp (the most a launch of any B uses)
    ql::KktLaunch P;
    std::memset(&P, 0, sizeof P);
    bool owned = false;
    if (int rc = launch_scratch(ds.kkt_scratch, stream, (size_t)ds.sm_count * per_sm * c.N * ql::KKT_FSTRIDE, &P.scratch,
                                &owned))
        return rc;
    P.c = c;
    P.jtab = ds.d_kkt_tab.get();
    P.htab = ds.d_kkt_tab.get() + c.nnz_true;
    P.io = *io;
    P.B = B;
    if (int rc = launch_kernel(ds, k, B, P, stream)) return rc;
    return end_scratch(P.scratch, owned, stream);
}

int check_kkt_factor(const Problem& p, int64_t B, const qlnlp_kkt_factor_io* io)
{
    const QlClass& c = p.cls;
    if (B < 0) return fail(QLNLP_EINVAL, "negative batch");
    if (!io || !io->hess || !io->jac || !io->dc || !io->factor || !io->status)
        return fail(QLNLP_EINVAL, "io, hess, jac, dc, factor and status are required");
    if (io->ldhess < ql_hess_nnz(c)) return fail(QLNLP_EINVAL, "ldhess %lld < nnz_hess %d", (long long)io->ldhess, ql_hess_nnz(c));
    if (io->ldjac < c.nnz_true) return fail(QLNLP_EINVAL, "ldjac %lld < nnz %d", (long long)io->ldjac, c.nnz_true);
    if (io->sx && io->ldsx < c.n_nlp) return fail(QLNLP_EINVAL, "ldsx %lld < n_nlp %d", (long long)io->ldsx, c.n_nlp);
    if (io->lddc < c.m_nlp) return fail(QLNLP_EINVAL, "lddc %lld < m_nlp %d", (long long)io->lddc, c.m_nlp);
    if (io->ldfactor < ql::kkt_factor_size(c))
        return fail(QLNLP_EINVAL, "ldfactor %lld < factor size %lld", (long long)io->ldfactor, ql::kkt_factor_size(c));
    for (const void* a : {(const void*)io->hess, (const void*)io->jac, (const void*)io->sx, (const void*)io->dc,
                          (const void*)io->factor})
        if ((reinterpret_cast<uintptr_t>(a) & 7) != 0) return fail(QLNLP_EINVAL, "arrays must be 8-byte aligned");
    if ((reinterpret_cast<uintptr_t>(io->status) & 3) != 0) return fail(QLNLP_EINVAL, "status must be 4-byte aligned");
    return QLNLP_OK;
}

int check_kkt_rhs(const Problem& p, int64_t R, const qlnlp_kkt_rhs_io* io)
{
    const QlClass& c = p.cls;
    if (R < 0) return fail(QLNLP_EINVAL, "negative batch");
    if (!io || !io->factor || !io->r1 || !io->r2 || !io->px || !io->pl || !io->status)
        return fail(QLNLP_EINVAL, "io, factor, r1, r2, px, pl and status are required");
    if (io->nfactor < 0) return fail(QLNLP_EINVAL, "negative nfactor");
    if (io->ldfactor < ql::kkt_factor_size(c))
        return fail(QLNLP_EINVAL, "ldfactor %lld < factor size %lld", (long long)io->ldfactor, ql::kkt_factor_size(c));
    if (io->ldr1 < c.n_nlp || io->ldpx < c.n_nlp)
        return fail(QLNLP_EINVAL, "ldr1 %lld / ldpx %lld < n_nlp %d", (long long)io->ldr1, (long long)io->ldpx, c.n_nlp);
    if (io->ldr2 < c.m_nlp || io->ldpl < c.m_nlp)
        return fail(QLNLP_EINVAL, "ldr2 %lld / ldpl %lld < m_nlp %d", (long long)io->ldr2, (long long)io->ldpl, c.m_nlp);
    for (const void* a : {(const void*)io->factor, (const void*)io->index, (const void*)io->r1, (const void*)io->r2,
                          (const void*)io->px, (const void*)io->pl})
        if ((reinterpret_cast<uintptr_t>(a) & 7) != 0) return fail(QLNLP_EINVAL, "arrays must be 8-byte aligned");
    if ((reinterpret_cast<uintptr_t>(io->status) & 3) != 0) return fail(QLNLP_EINVAL, "status must be 4-byte aligned");
    return QLNLP_OK;
}

int launch_kkt_factor(const Problem& p, DeviceState& ds, int64_t B, const qlnlp_kkt_factor_io* io, cudaStream_t stream)
{
    const QlClass& c = p.cls;
    if (int rc = ensure_kkt_tables(p, ds, stream)) return rc;
    ql::KktFactorLaunch P;
    std::memset(&P, 0, sizeof P);
    P.c = c;
    P.jtab = ds.d_kkt_tab.get();
    P.htab = ds.d_kkt_tab.get() + c.nnz_true;
    P.io = *io;
    P.B = B;
    return launch_kernel(ds, kkt_factor_spec(), B, P, stream);
}

int launch_kkt_solve_factored(const Problem& p, DeviceState& ds, int64_t R, const qlnlp_kkt_rhs_io* io, cudaStream_t stream)
{
    if (int rc = ensure_kkt_tables(p, ds, stream)) return rc;
    ql::KktSolveLaunch P;
    std::memset(&P, 0, sizeof P);
    P.c = p.cls;
    P.jtab = ds.d_kkt_tab.get();
    P.io = *io;
    P.B = R;
    return launch_kernel(ds, kkt_solve_factored_spec(), R, P, stream);
}

int check_kkt_residual(const Problem& p, int64_t B, const qlnlp_kkt_residual_io* io)
{
    const QlClass& c = p.cls;
    if (B < 0) return fail(QLNLP_EINVAL, "negative batch");
    if (!io || !io->hess || !io->jac || !io->dc || !io->r1 || !io->r2 || !io->px || !io->pl || !io->s1 || !io->s2)
        return fail(QLNLP_EINVAL, "io, hess, jac, dc, r1, r2, px, pl, s1 and s2 are required");
    const int64_t n = c.n_nlp, m = c.m_nlp;
    if (io->ldhess < ql_hess_nnz(c)) return fail(QLNLP_EINVAL, "ldhess %lld < nnz_hess %d", (long long)io->ldhess, ql_hess_nnz(c));
    if (io->ldjac < c.nnz_true) return fail(QLNLP_EINVAL, "ldjac %lld < nnz %d", (long long)io->ldjac, c.nnz_true);
    if (io->sx && io->ldsx < n) return fail(QLNLP_EINVAL, "ldsx %lld < n_nlp %lld", (long long)io->ldsx, (long long)n);
    if (io->ldr1 < n || io->ldpx < n || io->lds1 < n)
        return fail(QLNLP_EINVAL, "ldr1 %lld / ldpx %lld / lds1 %lld < n_nlp %lld", (long long)io->ldr1, (long long)io->ldpx,
                    (long long)io->lds1, (long long)n);
    if (io->lddc < m || io->ldr2 < m || io->ldpl < m || io->lds2 < m)
        return fail(QLNLP_EINVAL, "lddc %lld / ldr2 %lld / ldpl %lld / lds2 %lld < m_nlp %lld", (long long)io->lddc,
                    (long long)io->ldr2, (long long)io->ldpl, (long long)io->lds2, (long long)m);
    for (const void* a : {(const void*)io->hess, (const void*)io->jac, (const void*)io->sx, (const void*)io->dc,
                          (const void*)io->r1, (const void*)io->r2, (const void*)io->px, (const void*)io->pl,
                          (const void*)io->s1, (const void*)io->s2})
        if ((reinterpret_cast<uintptr_t>(a) & 7) != 0) return fail(QLNLP_EINVAL, "arrays must be 8-byte aligned");
    return QLNLP_OK;
}

int launch_kkt_residual(const Problem& p, DeviceState& ds, int64_t B, const qlnlp_kkt_residual_io* io, cudaStream_t stream)
{
    const QlClass& c = p.cls;
    if (int rc = ensure_kkt_tables(p, ds, stream)) return rc;
    ql::KktResidualLaunch P;
    std::memset(&P, 0, sizeof P);
    P.c = c;
    P.jtab = ds.d_kkt_tab.get();
    P.htab = ds.d_kkt_tab.get() + c.nnz_true;
    P.io = *io;
    P.B = B;
    return launch_kernel(ds, kkt_residual_spec(), B, P, stream);
}

// A row of a single call: n doubles, copied in from `in` before the launch and / or back to `out` after it
struct Row {
    const double* in;
    double* out;
    int64_t n;
};

// One call on host pointers (the MOI callbacks other than the cached evaluation), on the single-evaluation stream of
// the handle's first device: the rows (at most 5) are copied into device slots, each padded to an even length ld[i],
// run(ds, slot, ld, stream) launches on them, and the outputs come back before the call returns.
template <typename RUN>
int single_call(qlnlp_handle h, std::initializer_list<Row> rows, const char* what, RUN run)
{
    DeviceState& ds = h->devs[0];
    DeviceGuard guard(ds.device);
    if (int rc = ensure_device(h->prob, ds)) return rc;
    const cudaStream_t s = ds.one.stream.get();
    double* slot[5];
    int64_t ld[5];
    size_t total = 0;
    int i = 0;
    for (const Row& r : rows) total += ld[i++] = (r.n + 1) & ~1;
    if (int rc = grow_scratch(ds.one.slots, total, &slot[0])) return rc;
    cudaError_t e = cudaSuccess;
    i = 0;
    for (const Row& r : rows) {
        if (i) slot[i] = slot[i - 1] + ld[i - 1];
        if (r.in && e == cudaSuccess) e = cudaMemcpyAsync(slot[i], r.in, sizeof(double) * r.n, cudaMemcpyHostToDevice, s);
        ++i;
    }
    int rc = e == cudaSuccess ? run(ds, slot, ld, s) : fail(QLNLP_ECUDA, "%s: %s", what, cudaGetErrorString(e));
    i = 0;
    for (const Row& r : rows) {
        if (rc == QLNLP_OK && r.out) {
            e = cudaMemcpyAsync(r.out, slot[i], sizeof(double) * r.n, cudaMemcpyDeviceToHost, s);
            if (e != cudaSuccess) rc = fail(QLNLP_ECUDA, "%s: %s", what, cudaGetErrorString(e));
        }
        ++i;
    }
    return finish(s, rc, what);
}

int reserve_lane(const Problem& p, HostLane& ln, int64_t cap)
{
    if (ln.cap >= cap) return QLNLP_OK;
    ln = HostLane{std::move(ln.stream), std::move(ln.done)};      // the old buffers go before the new ones are made
    const std::pair<DevPtr<double>*, int64_t> rows[] = {{&ln.Z, p.ldz_e}, {&ln.x0, QL_NX}, {&ln.xf, QL_NX}, {&ln.f, 1},
        {&ln.grad, p.ldgrad_e}, {&ln.g, p.ldg_e}, {&ln.jac, std::max(p.ldjac_e, p.ldv_e)}};
    for (auto& r : rows)
        if (int rc = device_alloc(*r.first, (size_t)(cap * r.second))) return rc;
    if (int rc = pinned_alloc(ln.stage, (size_t)(cap * p.ldv_e), cudaHostAllocDefault)) return rc;
    ln.cap = cap;
    return QLNLP_OK;
}

// rows of `width` doubles: host (ld_h) <-> device (ld_d)
cudaError_t copy_rows(void* dst, int64_t ld_dst, const void* src, int64_t ld_src, int64_t width, int64_t rows,
                      cudaMemcpyKind kind, cudaStream_t s)
{
    if (ld_dst == width && ld_src == width)
        return cudaMemcpyAsync(dst, src, sizeof(double) * width * rows, kind, s);
    return cudaMemcpy2DAsync(dst, sizeof(double) * ld_dst, src, sizeof(double) * ld_src, sizeof(double) * width, rows, kind, s);
}

// is [jac, jac + B rows) inside a registered output buffer, on a row boundary, with the registered row stride?
bool is_registered(const qlnlp_handle_s* h, const double* jac, int64_t ldjac, int64_t B)
{
    for (const Registration& r : h->regs) {
        if (ldjac != r.ld || jac < r.ptr) continue;
        const int64_t off = jac - r.ptr;
        if (off % r.ld == 0 && off / r.ld + B <= r.rows) return true;
    }
    return false;
}

// ---- host-pointer batches ------------------------------------------------------------------------------------
// Pipeline over up to MAX_LANES streams, `chunk` evaluations per stage: H2D of the decision vectors, one fused launch,
// D2H of f / grad / g straight into the caller's arrays.  The Jacobian rows cross PCIe as the VALS stream (only the
// value-dependent entries: 2,794 of the 32,161 SPARSE_BLOCK values at the default instance) into a pinned staging
// buffer; while the next chunks are in flight the device's worker pool assembles the caller's rows from the constant
// image of the pattern and those values (hostrows.cpp) -- every 64-byte line of a row, or, when the caller has
// registered the output buffer (qlnlp_host_output_register), only the lines that hold a value-dependent entry.
int eval_host_impl(qlnlp_handle h, int dev, int64_t B, const qlnlp_batch_io* io)
{
    const Problem& p = h->prob;
    DeviceState& ds = h->devs[(size_t)dev];
    const QlClass& c = p.cls;
    // Uniform chunks: chunk i is [i * chunk, min(B, (i + 1) * chunk)).  (Smaller chunks at either end measured no
    // consistent gain, profiles/r02_host_path.md: the D2H copies, not the fill, bound the pipeline.)
    const int64_t chunk = std::max<int64_t>(1, std::min<int64_t>(B, h->opt_host_chunk));
    const int64_t nchunks = (B + chunk - 1) / chunk;
    const int nlanes = (int)std::min<int64_t>(MAX_LANES, nchunks);
    for (int l = 0; l < nlanes; ++l)
        if (int rc = reserve_lane(p, ds.lanes[l], chunk)) return rc;
    const bool compact = io->jac && B >= COMPACT_MIN_B && !p.kin;      // kinematic rows: the rows come back as they are
    bool touched_only = false;
    if (compact) {
        if (int rc = ensure_plan(h)) return rc;
        if (int rc = ensure_pool(h, dev)) return rc;
        touched_only = is_registered(h, io->jac, io->ldjac, B);
    }
    const int nnz_b = batch_nnz(p);
    // Device-side leading dimensions.  Padded (even) rows give the kernel its TMA / 16-byte paths, but when the caller's
    // rows are tightly packed a padded device copy needs a PITCHED transfer (one DMA descriptor per 9.7 KB row: 36 GB/s
    // instead of 50+).  PCIe is what bounds this path, not the kernel: mirror the caller's packing.
    const int64_t ldz_d = (io->ldz == c.n_nlp) ? c.n_nlp : p.ldz_e;
    const int64_t ldgrad_d = (io->grad && io->ldgrad == c.n_nlp) ? c.n_nlp : p.ldgrad_e;
    const int m_out = m_rows(p);
    const int64_t ldg_d = (io->g && io->ldg == m_out) ? m_out : p.ldg_e;
    const int64_t ldjac_d = (io->jac && io->ldjac == nnz_b) ? nnz_b : p.ldjac_e;      // uncompacted rows only
    auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t_begin = now();

    auto enqueue = [&](int64_t i) -> int {
        const double t0 = now();
        HostLane& ln = ds.lanes[i % nlanes];
        const int64_t b0 = i * chunk, nb = std::min(chunk, B - b0);
        cudaStream_t s = ln.stream.get();
        CUDA_TRY(copy_rows(ln.Z.get(), ldz_d, io->Z + b0 * io->ldz, io->ldz, c.n_nlp, nb, cudaMemcpyHostToDevice, s));
        if (io->x0) CUDA_TRY(cudaMemcpyAsync(ln.x0.get(), io->x0 + b0 * QL_NX, sizeof(double) * nb * QL_NX, cudaMemcpyHostToDevice, s));
        if (io->xf) CUDA_TRY(cudaMemcpyAsync(ln.xf.get(), io->xf + b0 * QL_NX, sizeof(double) * nb * QL_NX, cudaMemcpyHostToDevice, s));
        qlnlp_batch_io d;
        std::memset(&d, 0, sizeof d);
        d.Z = ln.Z.get(); d.ldz = ldz_d;
        d.x0 = io->x0 ? ln.x0.get() : nullptr;
        d.xf = io->xf ? ln.xf.get() : nullptr;
        d.f = io->f ? ln.f.get() : nullptr;
        d.grad = io->grad ? ln.grad.get() : nullptr; d.ldgrad = ldgrad_d;
        d.g = io->g ? ln.g.get() : nullptr; d.ldg = ldg_d;
        d.jac = io->jac ? ln.jac.get() : nullptr; d.ldjac = compact ? p.ldv_e : ldjac_d;
        if (int rc = p.kin ? launch_kin(p, ds, nb, &d, s) : launch(p, ds, nb, &d, s, compact ? ql::JM_VALS : -1)) return rc;
        // the staged values go first: the row builder only waits for them, f / grad / g land in the caller's arrays
        // by DMA while it works (the lanes are synchronised before the call returns)
        if (compact) {
            CUDA_TRY(cudaMemcpyAsync(ln.stage.get(), ln.jac.get(), sizeof(double) * nb * p.ldv_e, cudaMemcpyDeviceToHost, s));
            CUDA_TRY(cudaEventRecord(ln.done.get(), s));
        }
        if (io->f) CUDA_TRY(cudaMemcpyAsync(io->f + b0, ln.f.get(), sizeof(double) * nb, cudaMemcpyDeviceToHost, s));
        if (io->grad) CUDA_TRY(copy_rows(io->grad + b0 * io->ldgrad, io->ldgrad, ln.grad.get(), ldgrad_d, c.n_nlp, nb, cudaMemcpyDeviceToHost, s));
        if (io->g) CUDA_TRY(copy_rows(io->g + b0 * io->ldg, io->ldg, ln.g.get(), ldg_d, m_out, nb, cudaMemcpyDeviceToHost, s));
        if (!compact && io->jac)
            CUDA_TRY(copy_rows(io->jac + b0 * io->ldjac, io->ldjac, ln.jac.get(), ldjac_d, nnz_b, nb, cudaMemcpyDeviceToHost, s));
        ds.stat_t_enqueue += now() - t0;
        return QLNLP_OK;
    };
    // Row assembly runs on the pool's workers while this thread keeps the device fed: chunk j is handed to the pool
    // as soon as its copies have landed and the pool is free; chunk i may be enqueued once chunk i - nlanes has been
    // assembled (its pinned stage is reused).
    int64_t enq = 0, handed = 0, built = 0;
    double t_build0 = 0;
    auto progress = [&](bool may_block) -> int {
        if (!compact) { handed = built = enq; return QLNLP_OK; }
        if (handed > built) {                                   // a build is running
            if (ds.pool->busy()) {
                if (!may_block) return QLNLP_OK;
                ds.pool->finish();
            }
            ++built;
            ds.stat_t_build += now() - t_build0;
        }
        if (handed == built && handed < enq) {
            HostLane& ln = ds.lanes[handed % nlanes];
            const double t0 = now();
            cudaError_t q = may_block ? cudaEventSynchronize(ln.done.get()) : cudaEventQuery(ln.done.get());
            ds.stat_t_wait += now() - t0;
            if (q == cudaErrorNotReady) return QLNLP_OK;
            if (q != cudaSuccess) return fail(QLNLP_ECUDA, "host pipeline: %s", cudaGetErrorString(q));
            const int64_t b0 = handed * chunk, nb = std::min(chunk, B - b0);
            double* rows = io->jac + b0 * io->ldjac;
            t_build0 = now();
            h->plan->build_async(ds.pool.get(), ln.stage.get(), p.ldv_e, rows, io->ldjac, nb, touched_only);
            ++handed;
            ds.stat_host_rows += nb;
            ds.stat_host_lines += nb * (touched_only ? h->plan->touched_lines((int)((reinterpret_cast<uintptr_t>(rows) >> 3) & 7))
                                                     : (h->plan->nnz() + 7) / 8);
        }
        return QLNLP_OK;
    };
    for (int64_t i = 0; i < nchunks; ++i) {
        while (compact && i - built >= nlanes)
            if (int rc = progress(true)) return rc;
        if (int rc = enqueue(i)) return rc;
        ++enq;
        if (int rc = progress(false)) return rc;
    }
    while (built < enq)
        if (int rc = progress(true)) return rc;
    const double t_sync = now();
    for (int l = 0; l < nlanes; ++l) CUDA_TRY(cudaStreamSynchronize(ds.lanes[l].stream.get()));
    ds.stat_t_wait += now() - t_sync;
    ds.stat_t_total += now() - t_begin;
    return QLNLP_OK;
}

int eval_host(qlnlp_handle h, int dev, int64_t B, const qlnlp_batch_io* io)
{
    const Problem& p = h->prob;
    DeviceState& ds = h->devs[(size_t)dev];
    if (B == 0) return QLNLP_OK;
    if (int rc = check_batch(p, B, io, nullptr, true)) return rc;
    DeviceGuard guard(ds.device);
    if (int rc = ensure_device(p, ds)) return rc;
    const int rc = eval_host_impl(h, dev, B, io);
    if (rc != QLNLP_OK) {
        // copies into caller-owned host memory (and out of the pinned stage) may still be in flight: finish them
        // before the caller gets its buffers back
        if (ds.pool) ds.pool->finish();
        for (auto& ln : ds.lanes) finish(ln.stream.get(), rc, "host pipeline");
        cudaGetLastError();
    }
    return rc;
}

// contiguous, balanced split of range(B): the first B % n shards get one extra (sharding.shard_bounds)
void shard_bounds(int64_t B, int n, int s, int64_t* lo, int64_t* hi)
{
    const int64_t q = B / n, r = B % n;
    *lo = s * q + std::min<int64_t>(s, r);
    *hi = *lo + q + (s < r ? 1 : 0);
}

qlnlp_batch_io shard_io(const QlClass&, const qlnlp_batch_io& io, int64_t lo)
{
    qlnlp_batch_io d = io;
    d.Z = io.Z + lo * io.ldz;
    if (io.x0) d.x0 = io.x0 + lo * QL_NX;
    if (io.xf) d.xf = io.xf + lo * QL_NX;
    if (io.f) d.f = io.f + lo;
    if (io.grad) d.grad = io.grad + lo * io.ldgrad;
    if (io.g) d.g = io.g + lo * io.ldg;
    if (io.jac) d.jac = io.jac + lo * io.ldjac;
    return d;
}

// ---- single evaluations -------------------------------------------------------------------------------------
enum { HAVE_F = 1, HAVE_GRAD = 2, HAVE_G = 4, HAVE_J = 8 };

int reserve_one(const Problem& p, OneEval& o)
{
    if (o.mx) return QLNLP_OK;
    o.o_grad = 2;
    o.o_g = o.o_grad + p.ldgrad_e;
    o.o_vals = o.o_g + p.ldg_e;
    o.total = o.o_vals + p.ldv_e;
    // One decision vector is latency-bound: with mapped pinned memory the kernel fetches x and stores its 41 KB of
    // results over PCIe itself, which saves the two copy calls.
    if (int rc = pinned_alloc(o.hx, (size_t)(p.ldz_e + o.total), cudaHostAllocMapped)) return rc;
    o.hout = o.hx.get() + p.ldz_e;
    void* dp = nullptr;
    CUDA_TRY(cudaHostGetDevicePointer(&dp, o.hx.get(), 0));
    o.mx = static_cast<double*>(dp);
    o.mout = o.mx + p.ldz_e;
    o.valid = false;
    return QLNLP_OK;
}

// One decision vector on host pointers.  Ipopt asks for f, grad f, g and the Jacobian values of an iterate in four
// separate callbacks (moi.jl:1-24): the first callback at a new x evaluates EVERYTHING with one launch (f, grad, g and
// the value-dependent Jacobian entries: one kernel that reads x from and writes its 41 KB of results to mapped pinned
// memory, see reserve_one) and keeps the results; the other callbacks at the same x (compared bit for bit, 9.7 KB) are
// served from that cache.  The Jacobian values are assembled in the caller's array from the constant image of the
// pattern + the cached entries.  Runs on the handle's first device.
int eval_one(qlnlp_handle h, const double* x, double* f, double* grad, double* g, double* vals)
{
    if (int rc = check_handle(h)) return rc;
    if (!x) return fail(QLNLP_EINVAL, "null x");
    const Problem& p = h->prob;
    const QlClass& c = p.cls;
    if (p.kin) {
        // kinematic rows: the plain route -- copy x in, evaluate what was asked for, copy it out (no x cache)
        return single_call(h, {{x, nullptr, c.n_nlp}, {nullptr, f, 1}, {nullptr, grad, c.n_nlp}, {nullptr, g, m_rows(p)},
                               {nullptr, vals, batch_nnz(p)}}, "single evaluation",
                           [&](DeviceState& ds, double* const* d, const int64_t* ld, cudaStream_t s) {
                               qlnlp_batch_io io;
                               std::memset(&io, 0, sizeof io);
                               io.Z = d[0]; io.ldz = ld[0];
                               io.f = f ? d[1] : nullptr;
                               io.grad = grad ? d[2] : nullptr; io.ldgrad = ld[2];
                               io.g = g ? d[3] : nullptr; io.ldg = ld[3];
                               io.jac = vals ? d[4] : nullptr; io.ldjac = ld[4];
                               return launch_kin(p, ds, 1, &io, s);
                           });
    }
    DeviceState& ds = h->devs[0];
    DeviceGuard guard(ds.device);
    if (int rc = ensure_device(p, ds)) return rc;
    OneEval& o = ds.one;
    if (int rc = reserve_one(p, o)) return rc;
    const bool hit = h->opt_x_cache && o.valid && std::memcmp(o.hx.get(), x, sizeof(double) * c.n_nlp) == 0;
    if (!hit) {
        o.valid = false;
        std::memcpy(o.hx.get(), x, sizeof(double) * c.n_nlp);
        cudaStream_t s = o.stream.get();
        qlnlp_batch_io d;
        std::memset(&d, 0, sizeof d);
        d.Z = o.mx; d.ldz = c.n_nlp;                                 // odd ld: plain (non-TMA) loads from host memory
        d.f = o.mout;
        d.grad = o.mout + o.o_grad; d.ldgrad = p.ldgrad_e;
        d.g = o.mout + o.o_g; d.ldg = p.ldg_e;
        d.jac = o.mout + o.o_vals; d.ldjac = p.ldv_e + 1;            // odd ld: plain stores into host memory
        if (int rc = launch(p, ds, 1, &d, s, ql::JM_VALS)) return rc;
        CUDA_TRY(cudaStreamSynchronize(s));
        o.valid = true;
    }
    if (f) *f = o.hout[0];
    if (grad) std::memcpy(grad, o.hout + o.o_grad, sizeof(double) * c.n_nlp);
    if (g) std::memcpy(g, o.hout + o.o_g, sizeof(double) * c.m_nlp);
    if (vals) {
        if (int rc = ensure_plan(h)) return rc;
        h->plan->build_rows(o.hout + o.o_vals, p.ldv_e, vals, h->plan->nnz(), 0, 1, false);
    }
    return QLNLP_OK;
}

// DENSE: evaluate SPARSE_BLOCK (+ the kinematic entries) into a scratch row, scatter it into the zeroed m x n grid
int eval_dense_jacobian(qlnlp_handle h, const double* x, double* vals)
{
    if (!x) return fail(QLNLP_EINVAL, "null x");
    const Problem& p = h->prob;
    const int m = m_rows(p), nz = batch_nnz(p);
    const int64_t dense_n = (int64_t)m * p.cls.n_nlp;
    return single_call(h, {{x, nullptr, p.cls.n_nlp}, {nullptr, vals, dense_n}, {nullptr, nullptr, nz}}, "dense Jacobian",
                       [&](DeviceState& ds, double* const* d, const int64_t* ld, cudaStream_t s) -> int {
                           if (!ds.d_dense_lin) {          // the position in the grid of every value
                               std::vector<long long> lin;
                               for (const BatchEntry& e : batch_pattern(p)) lin.push_back((e.v.row - 1) + (long long)m * (e.v.col - 1));
                               if (int rc = upload(ds.d_dense_lin, lin.data(), lin.size())) return rc;
                           }
                           qlnlp_batch_io io;
                           std::memset(&io, 0, sizeof io);
                           io.Z = d[0]; io.ldz = ld[0];
                           io.jac = d[2]; io.ldjac = ld[2];
                           if (int rc = p.kin ? launch_kin(p, ds, 1, &io, s) : launch(p, ds, 1, &io, s)) return rc;
                           CUDA_TRY(cudaMemsetAsync(d[1], 0, sizeof(double) * dense_n, s));
                           ql::scatter_dense_kernel<<<(nz + 255) / 256, 256, 0, s>>>(d[2], ds.d_dense_lin.get(), d[1], nz);
                           CUDA_TRY(cudaGetLastError());
                           return QLNLP_OK;
                       });
}

// The problem of `d` on the devices `devices[0 .. ndev)`, which share the host cores.
int create_one(const qlnlp_problem_desc* d, const int* devices, int ndev, int jac_mode, qlnlp_handle* out)
{
    qlnlp_handle h = new (std::nothrow) qlnlp_handle_s();
    if (!h) return fail(QLNLP_ENOMEM, "out of host memory");
    Problem& p = h->prob;
    static std::atomic<uint64_t> g_serial{0};
    p.serial = ++g_serial;
    ql_class_init(&p.cls, (int)d->N, (int)d->k_trans, (int)d->init_mode, d->model.g, d->model.mb, d->model.mf, d->model.lb);
    ql_class_finish(&p.cls);
    p.jac_mode = jac_mode & ~QLNLP_WITH_KINEMATICS;
    p.kin = (jac_mode & QLNLP_WITH_KINEMATICS) != 0;
    p.leg_reach = d->model.l1 + d->model.l2 + d->model.lb / 2;
    std::memcpy(p.x0xf, d->x0, sizeof d->x0);
    std::memcpy(p.x0xf + QL_NX, d->xf, sizeof d->xf);
    const QlClass& c = p.cls;
    const int N = c.N;
    p.npad = (N + 31) & ~31;
    p.cost.assign((size_t)QL_NCOST * p.npad, 0.0);
    for (int k = 0; k < N; ++k) {
        for (int i = 0; i < QL_NX; ++i) {
            p.cost[(size_t)i * p.npad + k] = d->Q[k * QL_NX + i];
            p.cost[(size_t)(15 + i) * p.npad + k] = d->q[k * QL_NX + i];
        }
        for (int i = 0; i < QL_NU; ++i) {
            p.cost[(size_t)(30 + i) * p.npad + k] = d->R[k * QL_NU + i];
            p.cost[(size_t)(35 + i) * p.npad + k] = d->r[k * QL_NU + i];
        }
        p.cost[(size_t)40 * p.npad + k] = d->c[k];
    }
    if (int rc = block_plan(c, p.block)) {
        delete h;
        return rc;
    }
    plan_segments(c, p.block, p.segs, p.seg_begin);
    p.rmb = 1.0 / c.mb;
    p.rmf = 1.0 / c.mf;
    p.rIb = 1.0 / c.Ib;
    p.fastdiv = !std::getenv("QLNLP_IEEE_DIV") &&     // env: force the IEEE-division kernels
                ql::fastdiv_is_exact(c.mb) && ql::fastdiv_is_exact(c.mf) && ql::fastdiv_is_exact(c.Ib) &&
                ql::fastdiv_is_exact(6.0);
    p.ldz_e = (c.n_nlp + 1) & ~1;
    p.ldgrad_e = p.ldz_e;
    p.ldg_e = (m_rows(p) + 1) & ~1;
    p.ldjac_e = (batch_nnz(p) + 1) & ~1;
    p.ldv_e = (c.nnz_vals + 1) & ~1;
    h->devs.resize((size_t)ndev);
    for (int i = 0; i < ndev; ++i) h->devs[(size_t)i].device = devices[i];
    *out = h;
    return QLNLP_OK;
}

int check_desc(const qlnlp_problem_desc* d, int jac_mode_flags)
{
    const int jac_mode = jac_mode_flags & ~QLNLP_WITH_KINEMATICS;
    if (d->N < 2 || d->N > QL_MAX_N) return fail(QLNLP_EINVAL, "N=%lld outside [2, 1024]", (long long)d->N);
    if (d->k_trans < 1 || d->k_trans > d->N) return fail(QLNLP_EINVAL, "k_trans=%lld outside [1, N]", (long long)d->k_trans);
    if (d->init_mode != 1 && d->init_mode != 2) return fail(QLNLP_EINVAL, "init_mode must be 1 or 2");
    if (jac_mode != QLNLP_JAC_SPARSE_BLOCK && jac_mode != QLNLP_JAC_DENSE && jac_mode != QLNLP_JAC_SPARSE_TRUE) return fail(QLNLP_EINVAL, "unknown jac_mode %d", jac_mode);
    if (!d->Q || !d->R || !d->q || !d->r || !d->c) return fail(QLNLP_EINVAL, "cost tables are required");
    return QLNLP_OK;
}

// ---------------------------------------------------------------------------- device output allocator
// The driver's virtual-memory calls, reached through the runtime so that the library does not link libcuda.
struct DriverVmm {
    bool ok = false;
    PFN_cuDeviceGetAttribute_v2000 attr = nullptr;
    PFN_cuMemGetAllocationGranularity_v10020 granularity = nullptr;
    PFN_cuMemCreate_v10020 create = nullptr;
    PFN_cuMemGetAllocationPropertiesFromHandle_v10020 props = nullptr;
    PFN_cuMemRelease_v10020 release = nullptr;
    PFN_cuMemAddressReserve_v10020 reserve = nullptr;
    PFN_cuMemAddressFree_v10020 addr_free = nullptr;
    PFN_cuMemMap_v10020 map = nullptr;
    PFN_cuMemUnmap_v10020 unmap = nullptr;
    PFN_cuMemSetAccess_v10020 access = nullptr;
};

const DriverVmm& driver_vmm()
{
    static const DriverVmm d = [] {
        DriverVmm v;
        auto get = [](const char* sym, int ver, auto& fn) {
            void* p = nullptr;
            cudaDriverEntryPointQueryResult q;
            if (cudaGetDriverEntryPointByVersion(sym, &p, ver, cudaEnableDefault, &q) != cudaSuccess ||
                q != cudaDriverEntryPointSuccess)
                p = nullptr;
            fn = reinterpret_cast<std::remove_reference_t<decltype(fn)>>(p);
            return p != nullptr;
        };
        v.ok = get("cuDeviceGetAttribute", 2000, v.attr) & get("cuMemGetAllocationGranularity", 10020, v.granularity) &
               get("cuMemCreate", 10020, v.create) & get("cuMemGetAllocationPropertiesFromHandle", 10020, v.props) &
               get("cuMemRelease", 10020, v.release) & get("cuMemAddressReserve", 10020, v.reserve) &
               get("cuMemAddressFree", 10020, v.addr_free) & get("cuMemMap", 10020, v.map) &
               get("cuMemUnmap", 10020, v.unmap) & get("cuMemSetAccess", 10020, v.access);
        cudaGetLastError();
        return v;
    }();
    return d;
}

// One qlnlp_device_alloc block.  The table is process-wide, so a block can be freed after its handle is destroyed.
struct DeviceBlock {
    int device;
    size_t bytes;                       // mapped length (rounded to the granularity) or the cudaMalloc request
    bool vmm;                           // cuMemCreate + cuMemMap; otherwise cudaMalloc
    bool compressible;
    CUmemGenericAllocationHandle mem;
};
std::mutex g_blocks_mu;
std::map<uintptr_t, DeviceBlock> g_blocks;
std::atomic<int> g_refuse_compressible{0};   // tests: the next n compressible requests are refused as the driver would

// cuMemCreate with generic compression on `device`, mapped read-write for that device.  Returns false (and leaves
// nothing behind) whenever the driver declines: compressible backing is a limited resource, so a refusal is normal.
bool compressible_alloc(int device, size_t bytes, void** out, DeviceBlock& blk)
{
    const DriverVmm& d = driver_vmm();
    if (!d.ok) return false;
    if (g_refuse_compressible.load() > 0 && g_refuse_compressible.fetch_sub(1) > 0) return false;
    int vmm = 0, comp = 0;
    if (d.attr(&vmm, CU_DEVICE_ATTRIBUTE_VIRTUAL_MEMORY_MANAGEMENT_SUPPORTED, device) != CUDA_SUCCESS || !vmm) return false;
    if (d.attr(&comp, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, device) != CUDA_SUCCESS || !comp) return false;
    CUmemAllocationProp prop = {};
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = device;
    prop.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
    size_t gran = 0;
    if (d.granularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED) != CUDA_SUCCESS || gran == 0) return false;
    const size_t len = (bytes + gran - 1) / gran * gran;
    CUmemGenericAllocationHandle mem = 0;
    if (d.create(&mem, len, &prop, 0) != CUDA_SUCCESS) return false;
    CUmemAllocationProp got = {};
    CUdeviceptr va = 0;
    bool mapped = false;
    bool ok = d.props(&got, mem) == CUDA_SUCCESS && got.allocFlags.compressionType == CU_MEM_ALLOCATION_COMP_GENERIC &&
              d.reserve(&va, len, gran, 0, 0) == CUDA_SUCCESS;
    if (ok) ok = mapped = d.map(va, len, 0, mem, 0) == CUDA_SUCCESS;
    if (ok) {
        // read-write for the owning device and, as cudaMalloc memory would be, for every device that can reach it
        // peer to peer; if the driver refuses the peers, the owner alone
        std::vector<CUmemAccessDesc> acc(1);
        acc[0].location = prop.location;
        acc[0].flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) != cudaSuccess) ndev = 0;
        for (int peer = 0; peer < ndev; ++peer) {
            int can = 0;
            if (peer != device && cudaDeviceCanAccessPeer(&can, peer, device) == cudaSuccess && can) {
                CUmemAccessDesc a = acc[0];
                a.location.id = peer;
                acc.push_back(a);
            }
        }
        cudaGetLastError();
        ok = d.access(va, len, acc.data(), acc.size()) == CUDA_SUCCESS ||
             (acc.size() > 1 && d.access(va, len, acc.data(), 1) == CUDA_SUCCESS);
    }
    if (!ok) {
        if (mapped) d.unmap(va, len);
        if (va) d.addr_free(va, len);
        d.release(mem);
        return false;
    }
    blk = DeviceBlock{device, len, true, true, mem};
    *out = reinterpret_cast<void*>(va);
    return true;
}

// A block on `device`: compressible where offered and asked for, otherwise cudaMalloc.  Recorded in the block table.
int device_block_alloc(int device, size_t bytes, bool compressible, void** out)
{
    DeviceGuard guard(device);
    void* p = nullptr;
    DeviceBlock blk{device, bytes, false, false, 0};
    if (!(compressible && compressible_alloc(device, bytes, &p, blk))) {
        blk = DeviceBlock{device, bytes, false, false, 0};
        const cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) return alloc_failed(e, "cudaMalloc", bytes);
    }
    std::lock_guard<std::mutex> lk(g_blocks_mu);
    g_blocks[reinterpret_cast<uintptr_t>(p)] = blk;
    *out = p;
    return QLNLP_OK;
}

}  // namespace

// =============================================================================== C ABI
extern "C" {

int qlnlp_version(void) { return QLNLP_VERSION; }

const char* qlnlp_last_error(void) { return g_err.c_str(); }

int qlnlp_create(const qlnlp_problem_desc* d, int device, int jac_mode, qlnlp_handle* out)
{
    if (!d || !out) return fail(QLNLP_EINVAL, "null argument");
    *out = nullptr;
    if (int rc = check_desc(d, jac_mode)) return rc;
    return create_one(d, &device, 1, jac_mode, out);
}

int qlnlp_create_multi(const qlnlp_problem_desc* d, const int* devices, int ndev, int jac_mode, qlnlp_handle* out)
{
    if (!d || !out || !devices) return fail(QLNLP_EINVAL, "null argument");
    *out = nullptr;
    if (ndev < 1 || ndev > 64) return fail(QLNLP_EINVAL, "ndev=%d outside [1, 64]", ndev);
    for (int i = 0; i < ndev; ++i)
        for (int j = 0; j < i; ++j)
            if (devices[i] == devices[j]) return fail(QLNLP_EINVAL, "device %d listed twice", devices[i]);
    if (int rc = check_desc(d, jac_mode)) return rc;
    if (int rc = create_one(d, devices, ndev, jac_mode, out)) return rc;
    (*out)->multi = true;
    for (int i = 0; i < ndev; ++i) (*out)->drivers.emplace_back(new qlhost::Worker());
    return QLNLP_OK;
}

int qlnlp_destroy(qlnlp_handle h)
{
    if (!h) return QLNLP_OK;
    for (auto& w : h->drivers) w->wait();
    h->drivers.clear();
    for (DeviceState& ds : h->devs) {
        if (!ds.ready) continue;       // nothing on the device: a failed set-up releases what it made
        DeviceGuard guard(ds.device);
        cudaDeviceSynchronize();       // launches on caller streams may still use the handle's tables and counters
        ds = DeviceState();
    }
    delete h;
    return QLNLP_OK;
}

int qlnlp_dims(qlnlp_handle h, int64_t* n_nlp, int64_t* m_nlp, int64_t* nnz, int64_t* nnz_block)
{
    if (int rc = check_handle(h)) return rc;
    const Problem& p = h->prob;
    if (n_nlp) *n_nlp = p.cls.n_nlp;
    if (m_nlp) *m_nlp = m_rows(p);
    if (nnz) *nnz = (p.jac_mode == QLNLP_JAC_DENSE) ? (int64_t)m_rows(p) * p.cls.n_nlp : batch_nnz(p);
    if (nnz_block) *nnz_block = p.cls.nnz + (p.kin ? 8 * p.cls.N : 0);
    return QLNLP_OK;
}

int qlnlp_devices(qlnlp_handle h, int* devices, int cap, int* ndev)
{
    if (int rc = check_handle(h)) return rc;
    const int n = (int)h->devs.size();
    if (ndev) *ndev = n;
    if (devices)
        for (int i = 0; i < n && i < cap; ++i) devices[i] = h->devs[(size_t)i].device;
    return QLNLP_OK;
}

int qlnlp_shard_bounds(int64_t B, int nshards, int shard, int64_t* lo, int64_t* hi)
{
    if (B < 0 || nshards < 1 || shard < 0 || shard >= nshards || !lo || !hi) return fail(QLNLP_EINVAL, "bad shard arguments");
    shard_bounds(B, nshards, shard, lo, hi);
    return QLNLP_OK;
}

int qlnlp_jacobian_structure(qlnlp_handle h, int64_t* rows, int64_t* cols)
{
    if (int rc = check_handle(h)) return rc;
    if (!rows || !cols) return fail(QLNLP_EINVAL, "null output");
    const Problem& p = h->prob;
    if (p.jac_mode == QLNLP_JAC_DENSE) {
        // vec(Tuple.(CartesianIndices(zeros(m, n)))): column-major, row fastest (moi.jl:31-33)
        int64_t n = 0;
        for (int64_t col = 1; col <= p.cls.n_nlp; ++col)
            for (int64_t row = 1; row <= m_rows(p); ++row) { rows[n] = row; cols[n] = col; ++n; }
    } else {
        for (const BatchEntry& e : batch_pattern(p)) { *rows++ = e.v.row; *cols++ = e.v.col; }
    }
    return QLNLP_OK;
}

int qlnlp_constraint_bounds(qlnlp_handle h, double* lb, double* ub)
{
    if (int rc = check_handle(h)) return rc;
    if (!lb || !ub) return fail(QLNLP_EINVAL, "null output");
    const Problem& p = h->prob;
    for (int i = 0; i < m_rows(p); ++i) { lb[i] = 0.0; ub[i] = 0.0; }            // nlp.jl:66-67
    for (int i = 0; i < p.cls.N; ++i) ub[p.cls.c_body + i] = INFINITY;            // nlp.jl:69
    if (p.kin)                                                                    // nlp.jl:70 (commented out upstream)
        for (int i = 0; i < 2 * p.cls.N; ++i) ub[p.cls.m_nlp + i] = p.leg_reach;
    return QLNLP_OK;
}

int qlnlp_variable_bounds(qlnlp_handle h, double* xl, double* xu)
{
    if (int rc = check_handle(h)) return rc;
    if (!xl || !xu) return fail(QLNLP_EINVAL, "null output");
    const int N = h->prob.cls.N;
    const double half_pi = 3.14159265358979323846 / 2;
    for (int i = 0; i < h->prob.cls.n_nlp; ++i) { xl[i] = -INFINITY; xu[i] = INFINITY; }
    for (int k = 1; k <= N; ++k) {                                                // moi.jl:53-67, 1-based as written
        xl[3 + 20 * (k - 1) - 1] = -half_pi;
        xu[3 + 20 * (k - 1) - 1] = half_pi;
        if (k < N) {
            xl[20 + 20 * (k - 1) - 1] = 0.001;
            xu[20 + 20 * (k - 1) - 1] = 0.02;
            xl[22 + 20 * (k - 1) - 1] = 0.0;      // "lower bound of F": these hit yb / x1 of knot k+1, as in the reference
            xl[24 + 20 * (k - 1) - 1] = 0.0;
        }
    }
    return QLNLP_OK;
}

int qlnlp_set_option(qlnlp_handle h, const char* name, int64_t value)
{
    if (int rc = check_handle(h)) return rc;
    if (!name) return fail(QLNLP_EINVAL, "null option name");
    const std::string n(name);
    if (n == "host_chunk") { if (value < 1) return fail(QLNLP_EINVAL, "host_chunk must be >= 1"); h->opt_host_chunk = value; }
    else if (n == "host_threads") { if (value < 0) return fail(QLNLP_EINVAL, "host_threads must be >= 0"); h->opt_host_threads = value; }
    else if (n == "pin_threads") h->opt_pin_threads = value != 0;
    else if (n == "x_cache") { h->opt_x_cache = value != 0; h->devs[0].one.valid = false; }
    else if (n == "compressible") h->opt_compressible = value != 0;
    else return fail(QLNLP_EINVAL, "unknown option '%s'", name);
    if (n == "host_threads" || n == "pin_threads")          // the pools take both when they are made
        for (DeviceState& ds : h->devs) ds.pool.reset();
    return QLNLP_OK;
}

int qlnlp_eval_batch_device(qlnlp_handle h, int64_t B, const qlnlp_batch_io* io, void* stream)
{
    if (int rc = check_handle(h)) return rc;
    if (h->multi) return fail(QLNLP_EINVAL, "multi-device handle: use qlnlp_eval_batch_device_multi");
    if (B == 0) return QLNLP_OK;
    if (int rc = check_batch(h->prob, B, io, nullptr)) return rc;
    DeviceState& ds = h->devs[0];
    DeviceGuard guard(ds.device);
    if (int rc = ensure_device(h->prob, ds, static_cast<cudaStream_t>(stream))) return rc;
    if (h->prob.kin) return launch_kin(h->prob, ds, B, io, static_cast<cudaStream_t>(stream));
    return launch(h->prob, ds, B, io, static_cast<cudaStream_t>(stream));
}

int qlnlp_eval_batch_device_multi(qlnlp_handle h, const int64_t* B, const qlnlp_batch_io* io, void* const* streams)
{
    if (int rc = check_handle(h)) return rc;
    if (!B || !io) return fail(QLNLP_EINVAL, "null argument");
    const Problem& p = h->prob;
    for (size_t i = 0; i < h->devs.size(); ++i)
        if (B[i] != 0)
            if (int rc = check_batch(p, B[i], io + i, nullptr)) return rc;
    for (size_t i = 0; i < h->devs.size(); ++i) {
        DeviceState& ds = h->devs[i];
        if (B[i] == 0) continue;
        DeviceGuard guard(ds.device);
        cudaStream_t st = streams ? static_cast<cudaStream_t>(streams[i]) : nullptr;
        if (int rc = ensure_device(p, ds, st)) return rc;
        if (int rc = p.kin ? launch_kin(p, ds, B[i], io + i, st) : launch(p, ds, B[i], io + i, st)) return rc;
    }
    return QLNLP_OK;
}

int qlnlp_synchronize(qlnlp_handle h)
{
    if (int rc = check_handle(h)) return rc;
    for (const DeviceState& ds : h->devs) {
        if (!ds.ready) continue;
        DeviceGuard guard(ds.device);
        CUDA_TRY(cudaDeviceSynchronize());
    }
    return QLNLP_OK;
}

int qlnlp_eval_ragged_device(qlnlp_handle h, int64_t B, const qlnlp_batch_io* io, const qlnlp_ragged_io* rg, void* stream)
{
    if (int rc = check_handle(h)) return rc;
    if (h->multi) return fail(QLNLP_EINVAL, "multi-device handle: ragged launches take a single-device handle");
    if (!rg) return fail(QLNLP_EINVAL, "null ragged descriptor");
    if (h->prob.kin) return fail(QLNLP_EINVAL, "ragged launches do not carry the kinematic rows");
    if (B == 0) return QLNLP_OK;
    if (int rc = check_batch(h->prob, B, io, rg)) return rc;
    DeviceState& ds = h->devs[0];
    DeviceGuard guard(ds.device);
    if (int rc = ensure_device(h->prob, ds, static_cast<cudaStream_t>(stream))) return rc;
    const RagTable* table = nullptr;
    if (int rc = ragged_table(&h, 1, static_cast<cudaStream_t>(stream), &table)) return rc;
    return launch(h->prob, ds, B, io, static_cast<cudaStream_t>(stream), -1, rg, table, nullptr);
}

int qlnlp_eval_ragged_classes(const qlnlp_handle* hs, int ncls, int64_t B, const qlnlp_batch_io* io,
                              const qlnlp_ragged_io* rg, const int32_t* class_of, void* stream)
{
    if (!hs || ncls < 1 || ncls > 4096) return fail(QLNLP_EINVAL, "bad class list");
    if (!rg) return fail(QLNLP_EINVAL, "null ragged descriptor");
    if (ncls > 1 && !class_of) return fail(QLNLP_EINVAL, "class_of is required with more than one class");
    for (int i = 0; i < ncls; ++i) {
        if (int rc = check_handle(hs[i])) return rc;
        if (hs[i]->multi) return fail(QLNLP_EINVAL, "multi-device handle: ragged launches take single-device handles");
        if (hs[i]->devs[0].device != hs[0]->devs[0].device) return fail(QLNLP_EINVAL, "the classes of a ragged launch must share one device");
        if (batch_jm(hs[i]->prob) != batch_jm(hs[0]->prob)) return fail(QLNLP_EINVAL, "the classes of a ragged launch must share one Jacobian pattern");
        if (hs[i]->prob.kin) return fail(QLNLP_EINVAL, "ragged launches do not carry the kinematic rows");
    }
    if (B == 0) return QLNLP_OK;
    if (int rc = check_batch(hs[0]->prob, B, io, rg)) return rc;
    DeviceGuard guard(hs[0]->devs[0].device);
    for (int i = 0; i < ncls; ++i)
        if (int rc = ensure_device(hs[i]->prob, hs[i]->devs[0], static_cast<cudaStream_t>(stream))) return rc;
    const RagTable* table = nullptr;
    if (int rc = ragged_table(hs, ncls, static_cast<cudaStream_t>(stream), &table)) return rc;
    return launch(hs[0]->prob, hs[0]->devs[0], B, io, static_cast<cudaStream_t>(stream), -1, rg, table, class_of);
}

int qlnlp_eval_batch_host(qlnlp_handle h, int64_t B, const qlnlp_batch_io* io)
{
    if (int rc = check_handle(h)) return rc;
    if (!h->multi) return eval_host(h, 0, B, io);
    if (B == 0) return QLNLP_OK;
    if (B < 0 || !io) return fail(QLNLP_EINVAL, "bad batch");
    // the drivers share the row plan: build it before any of them may need it
    if (io->jac && !h->prob.kin)
        if (int rc = ensure_plan(h)) return rc;
    // contiguous shards, one driver thread per device, no exchange between the devices
    const int n = (int)h->devs.size();
    std::vector<int> rcs(n, QLNLP_OK);
    std::vector<std::string> msgs(n);
    for (int i = 0; i < n; ++i) {
        int64_t lo, hi;
        shard_bounds(B, n, i, &lo, &hi);
        if (hi == lo) continue;
        const qlnlp_batch_io d = shard_io(h->prob.cls, *io, lo);
        h->drivers[i]->submit([h, d, lo, hi, i, &rcs, &msgs] {
            rcs[i] = eval_host(h, i, hi - lo, &d);
            if (rcs[i]) msgs[i] = g_err;        // g_err is per thread
        });
    }
    for (auto& w : h->drivers) w->wait();
    for (int i = 0; i < n; ++i)
        if (rcs[i]) return fail(rcs[i], "device %d: %s", h->devs[(size_t)i].device, msgs[i].c_str());
    return QLNLP_OK;
}

int qlnlp_host_output_register(qlnlp_handle h, double* jac, int64_t ldjac, int64_t B)
{
    if (int rc = check_handle(h)) return rc;
    if (!jac || B < 1) return fail(QLNLP_EINVAL, "bad buffer");
    if ((reinterpret_cast<uintptr_t>(jac) & 7) != 0) return fail(QLNLP_EINVAL, "jac must be 8-byte aligned");
    if (ldjac < batch_nnz(h->prob)) return fail(QLNLP_EINVAL, "ldjac < nnz");
    if (h->prob.kin) return fail(QLNLP_EINVAL, "registered output rows are not available with the kinematic rows");
    if (int rc = ensure_plan(h)) return rc;
    qlnlp_host_output_unregister(h, jac);
    h->regs.push_back({jac, ldjac, B});
    // the constant image is written once, by the first device's pool
    if (int rc = ensure_pool(h, 0)) return rc;
    h->plan->build(h->devs[0].pool.get(), nullptr, 0, jac, ldjac, B, false);
    return QLNLP_OK;
}

int qlnlp_host_output_unregister(qlnlp_handle h, double* jac)
{
    if (int rc = check_handle(h)) return rc;
    for (auto it = h->regs.begin(); it != h->regs.end();)
        it = (it->ptr == jac) ? h->regs.erase(it) : it + 1;
    return QLNLP_OK;
}

int qlnlp_host_pin(void* ptr, int64_t bytes)
{
    if (!ptr || bytes <= 0) return fail(QLNLP_EINVAL, "bad buffer");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(QLNLP_ENODEVICE, "no CUDA device available");
    CUDA_TRY(cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterPortable));
    return QLNLP_OK;
}

int qlnlp_host_unpin(void* ptr)
{
    if (!ptr) return fail(QLNLP_EINVAL, "bad buffer");
    CUDA_TRY(cudaHostUnregister(ptr));
    return QLNLP_OK;
}

/* Page-locked host memory on 2 MB pages where the kernel grants them (madvise MADV_HUGEPAGE): rows of 257 KB each
 * touch 63 small pages, and on a virtualised host the page walks of a row builder that hops from line to line cost as
 * much as the stores.  The allocation is 2 MB aligned, zero-filled and registered with CUDA. */
int qlnlp_host_alloc(int64_t bytes, void** out)
{
    if (!out || bytes <= 0) return fail(QLNLP_EINVAL, "bad allocation request");
    *out = nullptr;
    const size_t huge = (size_t)2 << 20;
    const size_t len = ((size_t)bytes + huge - 1) / huge * huge;
    void* raw = mmap(nullptr, len + huge, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
    if (raw == MAP_FAILED) return fail(QLNLP_ENOMEM, "mmap of %zu bytes failed", len + huge);
    char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(raw) + huge - 1) / huge * huge);
    // give back the unaligned head and tail so that the mapping is exactly [base, base + len)
    if (base > (char*)raw) munmap(raw, (size_t)(base - (char*)raw));
    char* end = (char*)raw + len + huge;
    if (end > base + len) munmap(base + len, (size_t)(end - (base + len)));
#ifdef MADV_HUGEPAGE
    madvise(base, len, MADV_HUGEPAGE);        // best effort
#endif
    std::memset(base, 0, len);                // fault the pages in (as huge pages where possible) before pinning them
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) == cudaSuccess && ndev > 0) {
        cudaError_t e = cudaHostRegister(base, len, cudaHostRegisterPortable);
        if (e != cudaSuccess) {
            munmap(base, len);
            return fail(QLNLP_ECUDA, "cudaHostRegister of %zu bytes: %s", len, cudaGetErrorString(e));
        }
    } else {
        cudaGetLastError();                   // no device: plain (unpinned) memory, still usable by the CPU-side tests
    }
    *out = base;
    return QLNLP_OK;
}

int qlnlp_host_free(void* ptr, int64_t bytes)
{
    if (!ptr) return QLNLP_OK;
    const size_t huge = (size_t)2 << 20;
    const size_t len = ((size_t)bytes + huge - 1) / huge * huge;
    if (cudaHostUnregister(ptr) != cudaSuccess) cudaGetLastError();
    munmap(ptr, len);
    return QLNLP_OK;
}

int qlnlp_device_alloc(qlnlp_handle h, int64_t bytes, void** out)
{
    if (int rc = check_handle(h)) return rc;
    if (!out || bytes <= 0) return fail(QLNLP_EINVAL, "bad allocation request");
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(QLNLP_ENODEVICE, "no CUDA device available");
    }
    int device = h->devs[0].device;
    if (h->multi) {                    // the caller's current device, which must be one of the handle's
        if (cudaGetDevice(&device) != cudaSuccess) return fail(QLNLP_ECUDA, "cudaGetDevice failed");
        if (std::none_of(h->devs.begin(), h->devs.end(), [&](const DeviceState& ds) { return ds.device == device; }))
            return fail(QLNLP_EINVAL, "current device %d is not one of the handle's devices", device);
    }
    if (device < 0 || device >= ndev) return fail(QLNLP_EINVAL, "device %d out of range (0..%d)", device, ndev - 1);
    return device_block_alloc(device, (size_t)bytes, h->opt_compressible != 0, out);
}

int qlnlp_device_free(void* ptr)
{
    if (!ptr) return QLNLP_OK;
    DeviceBlock blk;
    {
        std::lock_guard<std::mutex> lk(g_blocks_mu);
        auto it = g_blocks.find(reinterpret_cast<uintptr_t>(ptr));
        if (it == g_blocks.end()) return fail(QLNLP_EINVAL, "%p was not returned by qlnlp_device_alloc", ptr);
        blk = it->second;
        g_blocks.erase(it);
    }
    DeviceGuard guard(blk.device);
    if (!blk.vmm) {
        CUDA_TRY(cudaFree(ptr));
        return QLNLP_OK;
    }
    // cudaFree waits for the device's work; unmapping does not, so wait here as cudaFree would
    CUDA_TRY(cudaDeviceSynchronize());
    const DriverVmm& d = driver_vmm();
    const CUdeviceptr va = reinterpret_cast<CUdeviceptr>(ptr);
    if (d.unmap(va, blk.bytes) != CUDA_SUCCESS || d.addr_free(va, blk.bytes) != CUDA_SUCCESS || d.release(blk.mem) != CUDA_SUCCESS)
        return fail(QLNLP_ECUDA, "releasing the mapping of %p failed", ptr);
    return QLNLP_OK;
}

/* torch.cuda.CUDAPluggableAllocator entry points (evaluator.py): segments of the caching pool the Python layer draws
 * its outputs from, so that outputs are reused in stream order instead of being allocated and freed per call.  Not part
 * of the C ABI.  The pool frees a segment only when it releases its cache, with no work pending on it. */
void* qlnlp_pool_alloc(ssize_t bytes, int device, void* /*stream*/)
{
    void* p = nullptr;
    return (bytes > 0 && device_block_alloc(device, (size_t)bytes, true, &p) == QLNLP_OK) ? p : nullptr;
}

void qlnlp_pool_free(void* ptr, size_t /*bytes*/, int /*device*/, void* /*stream*/) { qlnlp_device_free(ptr); }

/* tests: the next n compressible requests are refused as the driver refuses them when compressible backing runs out */
int qlnlp_debug_refuse_compressible(int n)
{
    g_refuse_compressible.store(n < 0 ? 0 : n);
    return QLNLP_OK;
}

/* tests: the n-th device or pinned allocation of a handle from now fails as an out-of-memory cudaMalloc would (n < 0:
 * none); returns the allocations the previous setting still had to go (-1: none armed).  And the blocks handles own. */
int qlnlp_debug_fail_alloc(int n) { return (int)std::max<int64_t>(-1, g_fail_alloc.exchange(n < 0 ? -1 : n)); }
int qlnlp_debug_owned_blocks(void) { return g_owned_blocks.load(); }

int qlnlp_device_alloc_info(const void* ptr, int64_t info[3])
{
    if (!ptr || !info) return fail(QLNLP_EINVAL, "null argument");
    std::lock_guard<std::mutex> lk(g_blocks_mu);
    const uintptr_t a = reinterpret_cast<uintptr_t>(ptr);
    auto it = g_blocks.upper_bound(a);
    if (it == g_blocks.begin() || a >= std::prev(it)->first + std::prev(it)->second.bytes)
        return fail(QLNLP_EINVAL, "%p is not inside a qlnlp_device_alloc block", ptr);
    --it;
    info[0] = it->second.compressible ? 1 : 0;
    info[1] = it->second.device;
    info[2] = (int64_t)it->second.bytes;
    return QLNLP_OK;
}

/* ---- Lagrangian Hessian (SURVEY.md 8f N3).  No reference counterpart: src/moi.jl:26-28 offers [:Grad, :Jac]. ---- */
int qlnlp_hessian_nnz(qlnlp_handle h, int64_t* nnz)
{
    if (int rc = check_handle(h)) return rc;
    if (!nnz) return fail(QLNLP_EINVAL, "null output");
    *nnz = ql_hess_nnz(h->prob.cls);
    return QLNLP_OK;
}

int qlnlp_hessian_structure(qlnlp_handle h, int64_t* rows, int64_t* cols)
{
    if (int rc = check_handle(h)) return rc;
    if (!rows || !cols) return fail(QLNLP_EINVAL, "null output");
    hessian_structure(h->prob.cls, rows, cols);
    return QLNLP_OK;
}

int qlnlp_eval_hessian_batch_device(qlnlp_handle h, int64_t B, const double* Z, int64_t ldz, const double* sigma,
                                    const double* lambda, int64_t ldlambda, double* H, int64_t ldh, void* stream)
{
    if (int rc = check_handle(h)) return rc;
    if (h->multi) return fail(QLNLP_EINVAL, "multi-device handle: the Hessian takes a single-device handle");
    if (h->prob.kin) return fail(QLNLP_EINVAL, "the Hessian does not cover the kinematic rows");
    if (B == 0) return QLNLP_OK;
    if (int rc = check_hessian(h->prob, B, Z, ldz, lambda, ldlambda, H, ldh, ql_hess_nnz(h->prob.cls))) return rc;
    DeviceState& ds = h->devs[0];
    DeviceGuard guard(ds.device);
    if (int rc = ensure_device(h->prob, ds, static_cast<cudaStream_t>(stream))) return rc;
    return launch_hessian(h->prob, ds, B, Z, ldz, sigma, 1.0, lambda, ldlambda, H, ldh, static_cast<cudaStream_t>(stream));
}

int qlnlp_eval_hessian_lagrangian(qlnlp_handle h, const double* x, double sigma, const double* lambda, double* vals)
{
    if (int rc = check_handle(h)) return rc;
    if (!x || !lambda || !vals) return fail(QLNLP_EINVAL, "null argument");
    const Problem& p = h->prob;
    if (p.kin) return fail(QLNLP_EINVAL, "the Hessian does not cover the kinematic rows");
    const QlClass& c = p.cls;
    return single_call(h, {{x, nullptr, c.n_nlp}, {lambda, nullptr, c.m_nlp}, {nullptr, vals, ql_hess_nnz(c)}}, "Hessian",
                       [&](DeviceState& ds, double* const* d, const int64_t* ld, cudaStream_t s) {
                           return launch_hessian(p, ds, 1, d[0], ld[0], nullptr, sigma, d[1], ld[1], d[2], ld[2], s);
                       });
}

/* ---- matrix-free products (MOI :JacVec / :HessVec) ---- */
int qlnlp_eval_jacobian_products_batch_device(qlnlp_handle h, int64_t B, const qlnlp_batch_io* io,
                                              const qlnlp_product_io* pv, void* stream)
{
    if (int rc = check_handle(h)) return rc;
    if (h->multi) return fail(QLNLP_EINVAL, "multi-device handle: the Jacobian products take a single-device handle");
    if (B == 0) return QLNLP_OK;
    if (int rc = check_products(h->prob, B, io, pv)) return rc;
    DeviceState& ds = h->devs[0];
    DeviceGuard guard(ds.device);
    if (int rc = ensure_device(h->prob, ds, static_cast<cudaStream_t>(stream))) return rc;
    return launch_products(h->prob, ds, B, io, pv, static_cast<cudaStream_t>(stream));
}

int qlnlp_eval_hessian_product_batch_device(qlnlp_handle h, int64_t B, const double* Z, int64_t ldz, const double* sigma,
                                            const double* lambda, int64_t ldlambda, const double* V, int64_t ldv,
                                            double* HV, int64_t ldhv, void* stream)
{
    if (int rc = check_handle(h)) return rc;
    if (h->multi) return fail(QLNLP_EINVAL, "multi-device handle: the Hessian takes a single-device handle");
    if (h->prob.kin) return fail(QLNLP_EINVAL, "the Hessian does not cover the kinematic rows");
    if (B == 0) return QLNLP_OK;
    if (int rc = check_hess_products(h->prob, B, Z, ldz, lambda, ldlambda, V, ldv, HV, ldhv)) return rc;
    DeviceState& ds = h->devs[0];
    DeviceGuard guard(ds.device);
    if (int rc = ensure_device(h->prob, ds, static_cast<cudaStream_t>(stream))) return rc;
    return launch_hess_products(h->prob, ds, B, Z, ldz, sigma, 1.0, lambda, ldlambda, V, ldv, HV, ldhv,
                                static_cast<cudaStream_t>(stream));
}

/* ---- batched KKT solve (qlnlp_kkt.cuh) ---- */
// the handles every KKT entry point takes
static int check_kkt_handle(qlnlp_handle h)
{
    if (int rc = check_handle(h)) return rc;
    if (h->multi) return fail(QLNLP_EINVAL, "multi-device handle: the KKT solve takes a single-device handle");
    if (h->prob.kin) return fail(QLNLP_EINVAL, "the KKT solve does not cover the kinematic rows");
    if (h->prob.jac_mode != QLNLP_JAC_SPARSE_TRUE) return fail(QLNLP_EINVAL, "the KKT solve takes a SPARSE_TRUE handle");
    return QLNLP_OK;
}

int qlnlp_kkt_solve_batch_device(qlnlp_handle h, int64_t B, const qlnlp_kkt_io* io, void* stream)
{
    if (int rc = check_kkt_handle(h)) return rc;
    if (B == 0) return QLNLP_OK;
    if (int rc = check_kkt(h->prob, B, io)) return rc;
    DeviceState& ds = h->devs[0];
    DeviceGuard guard(ds.device);
    if (int rc = ensure_device(h->prob, ds, static_cast<cudaStream_t>(stream))) return rc;
    return launch_kkt(h->prob, ds, B, io, static_cast<cudaStream_t>(stream));
}

int qlnlp_kkt_factor_size(qlnlp_handle h, int64_t* doubles)
{
    if (int rc = check_kkt_handle(h)) return rc;
    if (!doubles) return fail(QLNLP_EINVAL, "null output");
    *doubles = ql::kkt_factor_size(h->prob.cls);
    return QLNLP_OK;
}

int qlnlp_kkt_factor_batch_device(qlnlp_handle h, int64_t B, const qlnlp_kkt_factor_io* io, void* stream)
{
    if (int rc = check_kkt_handle(h)) return rc;
    if (B == 0) return QLNLP_OK;
    if (int rc = check_kkt_factor(h->prob, B, io)) return rc;
    DeviceState& ds = h->devs[0];
    DeviceGuard guard(ds.device);
    if (int rc = ensure_device(h->prob, ds, static_cast<cudaStream_t>(stream))) return rc;
    return launch_kkt_factor(h->prob, ds, B, io, static_cast<cudaStream_t>(stream));
}

int qlnlp_kkt_solve_factored_batch_device(qlnlp_handle h, int64_t R, const qlnlp_kkt_rhs_io* io, void* stream)
{
    if (int rc = check_kkt_handle(h)) return rc;
    if (R == 0) return QLNLP_OK;
    if (int rc = check_kkt_rhs(h->prob, R, io)) return rc;
    DeviceState& ds = h->devs[0];
    DeviceGuard guard(ds.device);
    if (int rc = ensure_device(h->prob, ds, static_cast<cudaStream_t>(stream))) return rc;
    return launch_kkt_solve_factored(h->prob, ds, R, io, static_cast<cudaStream_t>(stream));
}

int qlnlp_kkt_residual_batch_device(qlnlp_handle h, int64_t B, const qlnlp_kkt_residual_io* io, void* stream)
{
    if (int rc = check_kkt_handle(h)) return rc;
    if (B == 0) return QLNLP_OK;
    if (int rc = check_kkt_residual(h->prob, B, io)) return rc;
    DeviceState& ds = h->devs[0];
    DeviceGuard guard(ds.device);
    if (int rc = ensure_device(h->prob, ds, static_cast<cudaStream_t>(stream))) return rc;
    return launch_kkt_residual(h->prob, ds, B, io, static_cast<cudaStream_t>(stream));
}

// J w (transpose: J' y) at x for one evaluation
static int jacobian_product_one(qlnlp_handle h, const double* x, const double* v, double* out, bool transpose)
{
    if (int rc = check_handle(h)) return rc;
    if (!x || !v || !out) return fail(QLNLP_EINVAL, "null argument");
    const Problem& p = h->prob;
    const int64_t n = p.cls.n_nlp, m = m_rows(p);
    return single_call(h, {{x, nullptr, n}, {v, nullptr, transpose ? m : n}, {nullptr, out, transpose ? n : m}}, "product",
                       [&](DeviceState& ds, double* const* d, const int64_t* ld, cudaStream_t s) {
                           qlnlp_batch_io io;
                           std::memset(&io, 0, sizeof io);
                           io.Z = d[0]; io.ldz = ld[0];
                           qlnlp_product_io pv;
                           std::memset(&pv, 0, sizeof pv);
                           if (transpose) { pv.y = d[1]; pv.ldy = ld[1]; pv.jty = d[2]; pv.ldjty = ld[2]; }
                           else { pv.w = d[1]; pv.ldw = ld[1]; pv.jw = d[2]; pv.ldjw = ld[2]; }
                           return launch_products(p, ds, 1, &io, &pv, s);
                       });
}

int qlnlp_eval_constraint_jacobian_product(qlnlp_handle h, const double* x, const double* w, double* jw)
{
    return jacobian_product_one(h, x, w, jw, false);
}

int qlnlp_eval_constraint_jacobian_transpose_product(qlnlp_handle h, const double* x, const double* y, double* jty)
{
    return jacobian_product_one(h, x, y, jty, true);
}

int qlnlp_eval_hessian_lagrangian_product(qlnlp_handle h, const double* x, const double* v, double sigma,
                                          const double* lambda, double* hv)
{
    if (int rc = check_handle(h)) return rc;
    if (!x || !v || !lambda || !hv) return fail(QLNLP_EINVAL, "null argument");
    const Problem& p = h->prob;
    if (p.kin) return fail(QLNLP_EINVAL, "the Hessian does not cover the kinematic rows");
    const int64_t n = p.cls.n_nlp;
    return single_call(h, {{x, nullptr, n}, {lambda, nullptr, p.cls.m_nlp}, {v, nullptr, n}, {nullptr, hv, n}}, "product",
                       [&](DeviceState& ds, double* const* d, const int64_t* ld, cudaStream_t s) {
                           return launch_hess_products(p, ds, 1, d[0], ld[0], nullptr, sigma, d[1], ld[1], d[2], ld[2],
                                                       d[3], ld[3], s);
                       });
}

/* Batched initial guesses on the device (SURVEY.md 8f N2; main.ipynb:181-196): Z[b] = the class guess `base` with the
 * first 14 states of knots 1..k_trans interpolated from x0[b] to the handle's terminal state.  All device pointers. */
int qlnlp_initial_guess_batch_device(qlnlp_handle h, int64_t B, const double* base, const double* x0, double* Z,
                                     int64_t ldz, void* stream)
{
    if (int rc = check_handle(h)) return rc;
    if (B == 0) return QLNLP_OK;
    if (B < 0 || !base || !x0 || !Z) return fail(QLNLP_EINVAL, "bad arguments");
    const QlClass& c = h->prob.cls;
    DeviceState& ds = h->devs[0];
    if (ldz < c.n_nlp) return fail(QLNLP_EINVAL, "ldz < n_nlp");
    DeviceGuard guard(ds.device);
    if (int rc = ensure_device(h->prob, ds, static_cast<cudaStream_t>(stream))) return rc;
    const long long total = (long long)B * c.n_nlp;
    const int threads = 256;
    ql::initial_guess_kernel<<<(unsigned)((total + threads - 1) / threads), threads, 0, static_cast<cudaStream_t>(stream)>>>(
        base, x0, ds.d_x0xf.get() + QL_NX, Z, ldz, B, c.n_nlp, c.k_trans);
    CUDA_TRY(cudaGetLastError());
    return QLNLP_OK;
}

int qlnlp_eval_all(qlnlp_handle h, const double* x, double* f, double* grad, double* g, double* vals)
{
    if (int rc = check_handle(h)) return rc;
    if (vals && h->prob.jac_mode == QLNLP_JAC_DENSE) {
        if (int rc = eval_one(h, x, f, grad, g, nullptr)) return rc;
        return eval_dense_jacobian(h, x, vals);
    }
    return eval_one(h, x, f, grad, g, vals);
}

int qlnlp_eval_objective(qlnlp_handle h, const double* x, double* f)
{
    if (!f) return fail(QLNLP_EINVAL, "null output");
    return eval_one(h, x, f, nullptr, nullptr, nullptr);
}

int qlnlp_eval_objective_gradient(qlnlp_handle h, const double* x, double* grad)
{
    if (!grad) return fail(QLNLP_EINVAL, "null output");
    return eval_one(h, x, nullptr, grad, nullptr, nullptr);
}

int qlnlp_eval_constraint(qlnlp_handle h, const double* x, double* g)
{
    if (!g) return fail(QLNLP_EINVAL, "null output");
    return eval_one(h, x, nullptr, nullptr, g, nullptr);
}

int qlnlp_eval_constraint_jacobian(qlnlp_handle h, const double* x, double* vals)
{
    if (int rc = check_handle(h)) return rc;
    if (!vals) return fail(QLNLP_EINVAL, "null output");
    if (h->prob.jac_mode != QLNLP_JAC_DENSE) return eval_one(h, x, nullptr, nullptr, nullptr, vals);
    return eval_dense_jacobian(h, x, vals);
}

int qlnlp_launch_info(qlnlp_handle h, int64_t info[5])
{
    if (int rc = check_handle(h)) return rc;
    if (!info) return fail(QLNLP_EINVAL, "null output");
    for (int i = 0; i < 5; ++i) info[i] = h->devs[0].last_launch[i];
    return QLNLP_OK;
}

int qlnlp_host_path_info(qlnlp_handle h, int64_t info[8])
{
    if (int rc = check_handle(h)) return rc;
    if (!info) return fail(QLNLP_EINVAL, "null output");
    if (int rc = ensure_plan(h)) return rc;
    int64_t rows = 0, lines = 0;
    for (const DeviceState& ds : h->devs) {
        rows += ds.stat_host_rows;
        lines += ds.stat_host_lines;
    }
    const DeviceState& d0 = h->devs[0];
    info[0] = d0.pool ? d0.pool->size() : 0;          // worker threads per device (0: pool not started yet)
    info[1] = h->prob.cls.nnz_vals;                   // doubles per evaluation that cross PCIe for the Jacobian
    info[2] = h->plan->nnz();                         // doubles per row of the batch pattern
    info[3] = h->plan->touched_lines(0);              // 64-byte lines rewritten per registered row (aligned row)
    info[4] = (h->plan->nnz() + 7) / 8;               // 64-byte lines per row
    info[5] = qlhost::RowPlan::have_avx512() ? 1 : 0;
    info[6] = rows;                                   // rows assembled so far
    info[7] = lines;                                  // lines written so far
    return QLNLP_OK;
}

/* seconds spent so far by host-pointer batches of the first device: [0] total, [1] enqueueing copies and launches,
 * [2] waiting for the device / PCIe, [3] assembling rows (not part of the public header: tools/e2e_probe.py) */
int qlnlp_debug_host_times(qlnlp_handle h, double out[4])
{
    if (int rc = check_handle(h)) return rc;
    const DeviceState& ds = h->devs[0];
    out[0] = ds.stat_t_total; out[1] = ds.stat_t_enqueue; out[2] = ds.stat_t_wait; out[3] = ds.stat_t_build;
    return QLNLP_OK;
}

/* Launch geometry arithmetic, checkable without a device: out[0] = dynamic shared memory a SPARSE_BLOCK launch asks for
 * so that per_sm CTAs fit on an SM but per_sm + 1 never do, out[1] = the carve-out percentage requested for per_sm such
 * CTAs (not part of the public header: tests/test_cabi_cpu.py) */
int qlnlp_debug_launch_geometry(int64_t smem_per_sm, int64_t smem_optin, int per_sm, int64_t smem, int64_t out[2])
{
    if (!out || smem_per_sm <= 0 || per_sm < 1 || smem < 0) return fail(QLNLP_EINVAL, "bad arguments");
    const size_t padded = padded_smem((size_t)smem_per_sm, (size_t)smem_optin, per_sm, (size_t)smem);
    out[0] = (int64_t)padded;
    out[1] = carveout_pct((size_t)per_sm * (padded + 1024), (size_t)smem_per_sm);
    return QLNLP_OK;
}

/* Test hooks (not part of the public header): let CPU tests check the integer logic without a GPU.
 * qlnlp_debug_segments: out[i*6 + {0..5}] = k0 nk start end tmpl buf(of the first evaluation). */
int qlnlp_debug_segments(qlnlp_handle h, int64_t* out, int64_t cap, int64_t* nseg)
{
    if (int rc = check_handle(h)) return rc;
    const std::vector<QlSeg>& segs = h->prob.segs;
    if (nseg) *nseg = (int64_t)segs.size();
    if (out) {
        for (size_t i = 0; i < segs.size() && (int64_t)i < cap; ++i) {
            const QlSeg& s = segs[i];
            int64_t* o = out + 6 * i;
            o[0] = s.k0; o[1] = s.nk; o[2] = s.start; o[3] = s.end; o[4] = s.tmpl; o[5] = ql_seg_buffer((unsigned)i);
        }
    }
    return QLNLP_OK;
}

/* position of every VALS element inside a row of the handle's batch pattern; returns the count through *n */
int qlnlp_debug_vals_map(qlnlp_handle h, int32_t* pos, int64_t cap, int64_t* n)
{
    if (int rc = check_handle(h)) return rc;
    std::vector<double> image;
    std::vector<int32_t> p;
    batch_image_and_vals_map(h->prob, image, p);
    if (n) *n = (int64_t)p.size();
    if (pos)
        for (size_t i = 0; i < p.size() && (int64_t)i < cap; ++i) pos[i] = p[i];
    return QLNLP_OK;
}

/* the host row builder alone (no device): rows of the batch pattern from VALS rows; threads <= 0: the handle's pool */
int qlnlp_debug_build_rows(qlnlp_handle h, const double* vals, int64_t ldv, double* jac, int64_t ldjac, int64_t rows,
                           int touched_only, int threads)
{
    if (int rc = check_handle(h)) return rc;
    if (int rc = ensure_plan(h)) return rc;
    if (threads == 1) { h->plan->build_rows(vals, ldv, jac, ldjac, 0, rows, touched_only != 0); return QLNLP_OK; }
    const bool async = threads < -1;           // negative: the workers-only path the host pipeline uses (Pool::start)
    if (async) threads = -threads;
    DeviceState& ds = h->devs[0];
    if (threads > 1) { h->opt_host_threads = threads; ds.pool.reset(); }
    if (int rc = ensure_pool(h, 0)) return rc;
    if (async) {
        h->plan->build_async(ds.pool.get(), vals, ldv, jac, ldjac, rows, touched_only != 0);
        ds.pool->finish();
    } else {
        h->plan->build(ds.pool.get(), vals, ldv, jac, ldjac, rows, touched_only != 0);
    }
    return QLNLP_OK;
}

}  // extern "C"
