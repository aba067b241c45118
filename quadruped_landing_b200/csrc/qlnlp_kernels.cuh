// qlnlp_kernels.cuh -- fused batched evaluator kernel for sm_100a (B200).
//
// One warp per trajectory (decision vector), one lane per knot, ceil(N/32) passes; one warp per
// CTA so warps never synchronise with each other.  Evaluations are handed out in index order through a
// global ticket counter (keeps the rows written at any moment in a narrow address window).  Per evaluation the warp
//   1. stages Z through shared memory with ONE TMA bulk load per decision vector
//      (cp.async.bulk.shared.global + mbarrier; plain cp.async when Z is not 16-byte aligned); the next
//      vector is prefetched while the last pass streams its Jacobian values,
//   2. evaluates, per lane, the quadratic stage cost + gradient (costs.jl:6-34), one RK4 step of
//      the hybrid dynamics and its defect (constraints.jl:6-41), the contact / final-force /
//      body-clearance rows (constraints.jl:48-113,154) and the value-dependent entries of the
//      15x20 RK4 Jacobian by forward-mode duals held in registers (rk4_dual_gen.h),
//   3. writes the gradient, then the dynamics defects, in place over its (dead) slice of the staged Z and
//      flushes each with coalesced full-sector stores (scattered 8-byte stores of the defects cost 11 %
//      of throughput in the A/B runs of profiles/r01_ablation.md); reduces the cost with warp shuffles,
//   4. streams the SPARSE_BLOCK Jacobian values: the value stream is a concatenation of per-knot
//      runs (layout.h) that are ~90 % structural constants, so each 1-2-knot segment lives in a
//      shared-memory image whose constants persist from one evaluation to the next; the owner
//      lanes patch only the value-dependent entries and one lane fires a TMA bulk store
//      (cp.async.bulk.global.shared::cta, SASS UBLKCP) of the whole 4-8 KB segment.
// With the SPARSE_TRUE pattern (JM == 2: only structural non-zeros, 4,840 instead of 32,161 values) there are no
// zeros to persist: every lane writes its knot's whole run into a per-pass staging buffer and the pass goes
// out as one bulk store.
// All arithmetic is fp64 with explicit round-to-nearest add/mul/div (no FMA contraction) in the
// reference's operation order, so f, g, grad and the Jacobian values are bit-identical to the CPU
// oracle (sin/cos aside); the cost is accumulated knot by knot in the reference's sequential order.
// Divisions by the model constants use fastdiv.h: q = a*r, q' = fma(fma(-q, b, a), r, q) with r = RN(1/b), the
// correctly rounded quotient (Markstein) in the domain |a| >= 2^-969, a*r finite.  Outside it q' can miss by an ulp
// (0 < |a| < 2^-969), is +0 for a = -0, and NaN where a*r overflows; fastdiv.h states this exactly and why the
// kernels do not guard it.  The host verifies the domain per divisor at create time on every binade and falls back
// to IEEE division (template parameter FASTDIV = false, or QLNLP_IEEE_DIV) otherwise.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/qlnlp.h"
#include "fastdiv.h"
#include "layout.h"
#include "qlnlp_kin.cuh"

#ifndef QL_TRUE_WARPS
#define QL_TRUE_WARPS 8      // resident-warp target of the SPARSE_TRUE / VALS instantiations (252 registers at 8)
#endif
#ifndef QL_NONE_WARPS
#define QL_NONE_WARPS 16     // resident-warp target (register cap: 128) of the instantiation without a Jacobian:
                             // 16 warps/SM give +23..28 % over 8 (f+grad+g / g only), 20+ spill and lose
#endif

namespace ql {

// ---------------------------------------------------------------- PTX helpers
__device__ __forceinline__ unsigned smem_addr(const void* p)
{
    return static_cast<unsigned>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void st_shared_f64(unsigned addr, double v)
{
    asm volatile("st.shared.f64 [%0], %1;" ::"r"(addr), "d"(v) : "memory");
}
__device__ __forceinline__ void st_shared_zero16(unsigned addr)
{
    asm volatile("st.shared.v2.f64 [%0], {%1, %1};" ::"r"(addr), "d"(0.0) : "memory");
}
__device__ __forceinline__ void cp_async_8(unsigned dst, const void* src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
// TMA bulk copy shared::cta -> global, tracked by the issuing thread's bulk async-group
__device__ __forceinline__ void bulk_store(void* gdst, unsigned ssrc, unsigned bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(ssrc), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read()
{
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// TMA bulk copy global -> shared::cta, completion signalled on an mbarrier
__device__ __forceinline__ void mbar_init(unsigned mbar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory");
}
__device__ __forceinline__ void bulk_load(unsigned sdst, const void* gsrc, unsigned bytes, unsigned mbar)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(sdst),
                 "l"(gsrc), "r"(bytes), "r"(mbar)
                 : "memory");
}
// ask L2 to fetch a row that a later TMA load will want (the ticket of the next evaluation is known early)
__device__ __forceinline__ void prefetch_l2(const void* gsrc, unsigned bytes)
{
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gsrc), "r"(bytes) : "memory");
}
// g / grad / f are written once and never re-read by the kernel.  SPARSE_BLOCK kernel: streaming stores (st.global.cs, +0.6 % over
// plain stores).  The compact-output kernels re-read the cost table through L1 all the time (46 % of those loads miss it, ncu):
// there the rows go out with L1::no_allocate (+1.2 % SPARSE_TRUE, +0.5 % f+grad+g, +1.5 % g only; -1 % on the SPARSE_BLOCK headline,
// hence the split; profiles/r02_kernel_ab.md)
template <bool NO_ALLOCATE>
__device__ __forceinline__ void gst(double* p, double v)
{
    if (NO_ALLOCATE) asm volatile("st.global.L1::no_allocate.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
    else __stcs(p, v);
}
template <bool NO_ALLOCATE>
__device__ __forceinline__ void gst(double2* p, double2 v)
{
    if (NO_ALLOCATE) asm volatile("st.global.L1::no_allocate.v2.f64 [%0], {%1, %2};" ::"l"(p), "d"(v.x), "d"(v.y) : "memory");
    else __stcs(p, v);
}
#define QL_GST(ptr, v) gst<JM != JM_BLOCK>((ptr), (v))
__device__ __forceinline__ void mbar_wait(unsigned mbar, unsigned parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "QL_WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra QL_DONE_%=;\n"
        "bra QL_WAIT_%=;\n"
        "QL_DONE_%=:\n"
        "}\n" ::"r"(mbar),
        "r"(parity)
        : "memory");
}
// make generic-proxy shared-memory writes visible to the async (TMA) proxy
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// model constants + their reciprocals; division by a constant, correctly rounded (fastdiv.h)
template <bool FAST>
struct Consts {
    double g, mb, mf, Ib, rmb, rmf, rIb;
    __device__ __forceinline__ static double div(double a, double b, double r)
    {
        if (FAST) return fastdiv(a, b, r);
        return __ddiv_rn(a, b);
    }
    __device__ __forceinline__ double div_mb(double a) const { return div(a, mb, rmb); }
    __device__ __forceinline__ double div_mf(double a) const { return div(a, mf, rmf); }
    __device__ __forceinline__ double div_Ib(double a) const { return div(a, Ib, rIb); }
    __device__ __forceinline__ double div_six(double a) const { return div(a, 6.0, 0.16666666666666666); }
};

}  // namespace ql

// generated RK4 + Jacobian code: explicit rounding, shared-memory patch stores
#define QL_ADD(a, b) __dadd_rn((a), (b))
#define QL_SUB(a, b) __dsub_rn((a), (b))
#define QL_MUL(a, b) __dmul_rn((a), (b))
#define QL_DIV_MB(a) K.div_mb(a)
#define QL_DIV_MF(a) K.div_mf(a)
#define QL_DIV_IB(a) K.div_Ib(a)
#define QL_DIV_SIX(a) K.div_six(a)
#define QL_FN __device__ __forceinline__
#define QL_ST(ptr, off, val) ql::st_shared_f64((ptr) + 8u * (off), (val))
#define QL_PADD(ptr, n) ((ptr) + 8u * (n))
#include "rk4_dual_gen.h"
#include "true_run.h"

namespace ql {

#define QL_NJ_MAX (QL_NJ_MODE1 > QL_NJ_MODE3 ? QL_NJ_MODE1 : QL_NJ_MODE3)

// One (N, k_trans, init_mode, model, cost table) class of a RAGGED launch: what `Launch` carries for a plain one.
struct QlRagClass {
    QlClass c;
    double rmb, rmf, rIb;
    const double* cost;
    const double* x0_def;
    const double* xf_def;
    const QlSeg* segs;
    const int* seg_begin;
    int npad;
    int nseg;
};
#define QL_RAGCLASS_BYTES 192
static_assert(sizeof(QlRagClass) <= QL_RAGCLASS_BYTES && QL_RAGCLASS_BYTES % 16 == 0, "QlRagClass does not fit its shared-memory slot");

struct Launch {
    QlClass c;                 // RAGGED launches: only c.N matters here (the LARGEST horizon, for the shared-memory layout)
    double rmb, rmf, rIb;      // RN(1/mb), RN(1/mf), RN(1/Ib)
    const double* cost;        // [QL_NCOST][npad] field-major: Q 0-14, q 15-29, R 30-34, r 35-39, c 40
    int npad;
    int nseg;
    const double* x0_def;      // [15]  desc.x0
    const double* xf_def;      // [15]  desc.xf
    const QlSeg* segs;         // segment plan, all passes
    const int* seg_begin;      // [npass + 1]
    qlnlp_batch_io io;         // the caller's arrays, as the entry point took them
    long long B;
    // RAGGED instantiation only: the b-th evaluation of the launch is problem index[b] (or b) of a flat, mixed-size
    // batch; its rows start at Z + z_off[i], grad + z_off[i], g + g_off[i], jac + j_off[i]; f, x0, xf are indexed by i
    const long long* index;
    const long long* z_off;
    const long long* g_off;
    const long long* j_off;
    const QlRagClass* classes; // RAGGED: per-class records; problem i belongs to class cls_of[i] (class 0 when cls_of is null)
    const int* cls_of;
    unsigned* ticket;          // [0] next evaluation to hand out, [1] CTAs that have finished (both 0 between launches)
    int bulk;                  // 1: jac rows are 16 B aligned -> TMA bulk stores
    int zbulk;                 // 1: Z rows are 16 B aligned and ldz > n_nlp -> one TMA bulk load per vector
};

// shared memory carve-up: staged Z (same layout as in HBM) | mbarrier | two J staging buffers | segment plan
__host__ __device__ inline int zbuf_len(int N) { return QL_NZK * N + 2; }     // n_nlp + 1 rounded up to even, + mbarrier
#define QL_FBUF 32           // per-lane cost terms of a pass, summed in knot order (costs.jl:9-15)
enum { JM_NONE = 0, JM_BLOCK = 1, JM_TRUE = 2, JM_VALS = 3,      // which Jacobian value stream the kernel produces
       JM_PROD = 4 };                                              // ... or J w / J' y instead of a stream (eval_prod_kernel)
#define QL_PROD_BUF 642      // doubles of the JM_PROD staging buffer: one pass of J' y (32 x 20), or of J w's defect rows + parity
static_assert(QL_VALS_LEN_MODE1 == QL_VALS_LEN_INIT && QL_VALS_LEN_MODE2 == QL_VALS_LEN_INIT &&
              QL_VALS_LEN_MODE1_JUMP == QL_VALS_LEN_JUMPK && QL_VALS_LEN_MODE2_JUMP == QL_VALS_LEN_JUMPK &&
              QL_VALS_LEN_MODE3 == QL_VALS_LEN_M3, "layout.h VALS run lengths out of date");
__host__ __device__ inline size_t smem_jregion_bytes(int N, int jm)
{
    const int nseg_max = (N + 1) / 2 + (N + QL_LANES - 1) / QL_LANES;
    if (jm == JM_BLOCK) return sizeof(double) * 2 * QL_JBUF + sizeof(QlSeg) * nseg_max;
    if (jm == JM_TRUE || jm == JM_VALS) return sizeof(double) * QL_TRUE_PBUF;
    if (jm == JM_PROD) return sizeof(double) * QL_PROD_BUF;
    return 0;
}
__host__ __device__ inline size_t smem_bytes(int N, int jm)
{
    return sizeof(double) * (size_t)(zbuf_len(N) + QL_FBUF) + QL_RAGCLASS_BYTES + smem_jregion_bytes(N, jm);
}

// Start fetching a decision vector into shared memory.  zbulk: one TMA bulk load of n+1 doubles (n is odd, the
// row is 16-byte aligned with ldz > n, so the extra element is in bounds); else coalesced 8-byte cp.async.
__device__ __forceinline__ void stage_z(const double* __restrict__ Zrow, unsigned zaddr, unsigned mbar, int n, int lane,
                                        bool zbulk)
{
    if (zbulk) {
        fence_proxy_async();        // order this warp's earlier generic accesses to zbuf before the async write
        __syncwarp();
        if (lane == 0) bulk_load(zaddr, Zrow, 8u * (unsigned)(n + 1), mbar);
    } else {
        for (int e = lane; e < n; e += QL_LANES) cp_async_8(zaddr + 8u * (unsigned)e, Zrow + e);
        cp_async_commit();
    }
}

// fsum + t[0] + t[1] + ... + t[31], strictly left to right (costs.jl:9-15); lanes without a knot have stored -0.0
__device__ __forceinline__ double f_chain(double fsum, const double* fbuf)
{
    // (forcing all 16 loads ahead of the adds with volatile asm changes nothing measurable: profiles/r02_kernel_ab.md)
    const double2* f2 = reinterpret_cast<const double2*>(fbuf);
#pragma unroll
    for (int s = 0; s < QL_LANES / 2; ++s) {
        const double2 t = f2[s];
        fsum = __dadd_rn(__dadd_rn(fsum, t.x), t.y);
    }
    return fsum;
}

// The Jacobian-product launch (JM_PROD): the Launch fields keep their meaning (io.jac must be null), the products'
// vectors and outputs come on top.  Rows are [B][ld]; a null w (or y) skips J w (or J' y).
struct ProdLaunch : Launch {
    qlnlp_product_io pv;                   // jw and y rows hold m_nlp + 2N entries with kinematic rows
    int kin;                               // 1: the handle's kinematic rows (rows m_nlp + 2(k-1) + foot) are part of J and g
};

// Matrix-free products of one knot (lane k) for JM_PROD, after steps 1-4 of the pass.  Every output entry is the left
// fold of entry * vector over the structurally non-zero entries of the SPARSE_TRUE pattern (rows of J w in ascending
// column order, columns of J' y in ascending row order), so the bits are those of a fold of the materialised values.
// Both outputs are staged in `jb` and leave with coalesced stores: the defect rows of J w at the destination's parity
// like the defects, J' y in the Z layout like the gradient.  w and y are read straight from global memory (L1): a
// staged copy of w next to the staged Z would not fit shared memory at the largest horizons.
template <bool FASTDIV>
__device__ __forceinline__ void prod_pass(const ProdLaunch& P, const QlClass& c, long long b, int p, int lane, int k,
                                          const double* xk, const double* jv, double jtheta, double* jb)
{
    const bool act = k <= c.N, has_u = k < c.N, jump = has_u && (k == c.k_trans - 1);
    const bool first_is_y1 = (c.init_mode == 1);
    const int mode = k >= c.k_trans ? 3 : c.init_mode;
    // kinematic rows (qlnlp_kin.cuh): d/d(xb, yb, x_foot, y_foot) = (dx, dy, -dx, -dy) / norm, IEEE division
    double kv[2][4];
    if (P.kin && act) {
#pragma unroll
        for (int f = 0; f < 2; ++f) {
            double dx, dy;
            const double n = kin_norm(xk, f, &dx, &dy);
            kv[f][0] = __ddiv_rn(dx, n);
            kv[f][1] = __ddiv_rn(dy, n);
            kv[f][2] = __ddiv_rn(-dx, n);
            kv[f][3] = __ddiv_rn(-dy, n);
            if (P.io.g) gst<true>(P.io.g + b * P.io.ldg + c.m_nlp + 2 * (k - 1) + f, n);
        }
    }
    if (P.pv.jw) {
        double* const jwrow = P.pv.jw + b * P.pv.ldjw;
        double* const ddst = jwrow + c.c_dyn + p * QL_LANES * QL_NX;
        const int dpar = (int)((reinterpret_cast<uintptr_t>(ddst) >> 3) & 1);
        __syncwarp();                                   // the previous flush has read jb
        if (act) {
            const double* const wk = P.pv.w + b * P.pv.ldw + (long long)QL_NZK * (k - 1);
            double wv[QL_NZK];
#pragma unroll
            for (int j = 0; j < QL_NZK; ++j) wv[j] = (j < QL_NX || has_u) ? __ldg(wk + j) : 0.0;
            if (k == 1)
#pragma unroll
                for (int i = 0; i < QL_NX; ++i) gst<true>(jwrow + i, wv[i]);                       // init rows
            if (k == c.N)
#pragma unroll
                for (int i = 0; i < QL_NX - 1; ++i) gst<true>(jwrow + c.c_term + i, wv[i]);        // term rows
            gst<true>(jwrow + c.c_cfirst + (k - 1), first_is_y1 ? wv[4] : wv[6]);
            if (k >= c.k_trans) gst<true>(jwrow + c.c_cother + (k - c.k_trans), first_is_y1 ? wv[6] : wv[4]);
            if (k == c.N - 1) gst<true>(jwrow + c.c_fctrl, __dadd_rn(wv[16], wv[18]));
            gst<true>(jwrow + c.c_body + (k - 1), __dadd_rn(wv[1], __dmul_rn(jtheta, wv[2])));
            if (P.kin) {
#pragma unroll
                for (int f = 0; f < 2; ++f) {
                    const int jx = f ? 5 : 3;
                    const double s = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(kv[f][0], wv[0]), __dmul_rn(kv[f][1], wv[1])),
                                                         __dmul_rn(kv[f][2], wv[jx])), __dmul_rn(kv[f][3], wv[jx + 1]));
                    gst<true>(jwrow + c.m_nlp + 2 * (k - 1) + f, s);
                }
            }
            if (has_u) {
                double wn[QL_NX], o[QL_NX];
#pragma unroll
                for (int i = 0; i < QL_NX; ++i) wn[i] = __ldg(wk + QL_NZK + i);
                if (mode == 3) ql_rk4_jvp_mode3(jv, wv, wn, o);
                else if (mode == 1) { if (jump) ql_rk4_jvp_mode1_jump(jv, wv, wn, o); else ql_rk4_jvp_mode1(jv, wv, wn, o); }
                else { if (jump) ql_rk4_jvp_mode2_jump(jv, wv, wn, o); else ql_rk4_jvp_mode2(jv, wv, wn, o); }
#pragma unroll
                for (int i = 0; i < QL_NX; ++i) jb[dpar + lane * QL_NX + i] = o[i];
            }
        }
        __syncwarp();
        // the defect rows of this pass, as in step 4
        const int k_first = p * QL_LANES + 1;
        const int ndyn = min(QL_LANES, c.N - k_first) * QL_NX;
        const int j0 = dpar, j1 = dpar + ndyn;
        const int a = (j0 + 1) & ~1, e = j1 & ~1;
        const double2* s2 = reinterpret_cast<const double2*>(jb);
        double2* d2 = reinterpret_cast<double2*>(ddst - dpar);
        for (int i = (a >> 1) + lane; i < (e >> 1); i += QL_LANES) gst<true>(d2 + i, s2[i]);
        if (lane == 0 && a > j0 && ndyn > 0) gst<true>(ddst, jb[j0]);
        if (lane == 1 && e < j1 && e >= a) gst<true>(ddst + (e - dpar), jb[e]);
    }
    if (P.pv.jty) {
        double* const jtyrow = P.pv.jty + b * P.pv.ldjty;
        __syncwarp();                                   // the J w flush has read jb
        if (act) {
            const double* const yr = P.pv.y + b * P.pv.ldy;
            double a[QL_NX], o[QL_NZK];
            // rows above the RK4 block in each state column: init (k = 1) or term (k = N), then knot k-1's -I block
#pragma unroll
            for (int j = 0; j < QL_NX; ++j) {
                if (k == 1) a[j] = __ldg(yr + j);
                else {
                    const double mi = -__ldg(yr + c.c_dyn + QL_NX * (k - 2) + j);
                    a[j] = (k == c.N && j < QL_NX - 1) ? __dadd_rn(__ldg(yr + c.c_term + j), mi) : mi;
                }
            }
            if (has_u) {
                double yd[QL_NX];
#pragma unroll
                for (int i = 0; i < QL_NX; ++i) yd[i] = __ldg(yr + c.c_dyn + QL_NX * (k - 1) + i);
                if (mode == 3) ql_rk4_vjp_mode3(jv, yd, a, o);
                else if (mode == 1) { if (jump) ql_rk4_vjp_mode1_jump(jv, yd, a, o); else ql_rk4_vjp_mode1(jv, yd, a, o); }
                else { if (jump) ql_rk4_vjp_mode2_jump(jv, yd, a, o); else ql_rk4_vjp_mode2(jv, yd, a, o); }
                if (k == c.N - 1) {                     // final-control row on F1y, F2y
                    const double yf = __ldg(yr + c.c_fctrl);
                    o[16] = __dadd_rn(o[16], yf);
                    o[18] = __dadd_rn(o[18], yf);
                }
            } else {
#pragma unroll
                for (int j = 0; j < QL_NX; ++j) o[j] = a[j];
#pragma unroll
                for (int j = QL_NX; j < QL_NZK; ++j) o[j] = 0.0;          // beyond n_nlp: not flushed
            }
            // the extra rows, in row order: contact-first / contact-other, body, kinematic
            const double yfirst = __ldg(yr + c.c_cfirst + (k - 1));
            const double yother = k >= c.k_trans ? __ldg(yr + c.c_cother + (k - c.k_trans)) : 0.0;
            if (first_is_y1) {
                o[4] = __dadd_rn(o[4], yfirst);
                if (k >= c.k_trans) o[6] = __dadd_rn(o[6], yother);
            } else {
                o[6] = __dadd_rn(o[6], yfirst);
                if (k >= c.k_trans) o[4] = __dadd_rn(o[4], yother);
            }
            const double ybody = __ldg(yr + c.c_body + (k - 1));
            o[1] = __dadd_rn(o[1], ybody);
            o[2] = __dadd_rn(o[2], __dmul_rn(jtheta, ybody));
            if (P.kin) {
                const double y0 = __ldg(yr + c.m_nlp + 2 * (k - 1)), y1 = __ldg(yr + c.m_nlp + 2 * (k - 1) + 1);
                o[0] = __dadd_rn(__dadd_rn(o[0], __dmul_rn(kv[0][0], y0)), __dmul_rn(kv[1][0], y1));
                o[1] = __dadd_rn(__dadd_rn(o[1], __dmul_rn(kv[0][1], y0)), __dmul_rn(kv[1][1], y1));
                o[3] = __dadd_rn(o[3], __dmul_rn(kv[0][2], y0));
                o[4] = __dadd_rn(o[4], __dmul_rn(kv[0][3], y0));
                o[5] = __dadd_rn(o[5], __dmul_rn(kv[1][2], y1));
                o[6] = __dadd_rn(o[6], __dmul_rn(kv[1][3], y1));
            }
            double2* const jb2 = reinterpret_cast<double2*>(jb + lane * QL_NZK);
#pragma unroll
            for (int j = 0; j < QL_NZK / 2; ++j) jb2[j] = make_double2(o[2 * j], o[2 * j + 1]);
        }
        __syncwarp();
        // this pass's columns, as the gradient flush
        const int e0 = p * QL_LANES * QL_NZK;
        const int cnt = min(QL_LANES * QL_NZK, c.n_nlp - e0);
        if ((reinterpret_cast<uintptr_t>(jtyrow) & 15) == 0) {
            const double2* s2 = reinterpret_cast<const double2*>(jb);
            double2* d2 = reinterpret_cast<double2*>(jtyrow + e0);
            for (int i = lane; i < (cnt >> 1); i += QL_LANES) gst<true>(d2 + i, s2[i]);
            if ((cnt & 1) && lane == 0) gst<true>(jtyrow + e0 + cnt - 1, jb[cnt - 1]);
        } else {
            for (int i = lane; i < cnt; i += QL_LANES) gst<true>(jtyrow + e0 + i, jb[i]);
        }
    }
}


template <int JM, bool FASTDIV, bool RAGGED>
__global__ void __launch_bounds__(QL_LANES, JM == JM_NONE ? QL_NONE_WARPS : (JM == JM_BLOCK ? 8 : QL_TRUE_WARPS)) eval_kernel(const __grid_constant__ Launch P)
{
#include "qlnlp_eval_body.cuh"
}

// J w and / or J' y (with f, grad f, g as requested) of B decision vectors: the evaluator's steps 1-4, then prod_pass
template <bool FASTDIV>
__global__ void __launch_bounds__(QL_LANES, QL_TRUE_WARPS) eval_prod_kernel(const __grid_constant__ ProdLaunch P)
{
    constexpr int JM = JM_PROD;
    constexpr bool RAGGED = false;
#include "qlnlp_eval_body.cuh"
}

// Initial guesses of a sweep (main.ipynb:181-196, cell 7): every problem's guess is the class guess `base` except the
// first 14 states of knots 1..k_trans, which interpolate from the problem's own initial state to the terminal state:
//   Xguess[k] = xinit + (xterm - xinit) / (k_trans - 1) * (k - 1)          (evaluated left to right, like the notebook)
// One thread per element of Z; rows of Z are ldz apart.
__global__ void initial_guess_kernel(const double* __restrict__ base, const double* __restrict__ x0, const double* __restrict__ xterm,
                                     double* __restrict__ Z, long long ldz, long long B, int n_nlp, int k_trans)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= B * n_nlp) return;
    const long long b = t / n_nlp;
    const int e = (int)(t - b * n_nlp);
    const int k = e / QL_NZK + 1, i = e - (k - 1) * QL_NZK;
    double v = __ldg(base + e);
    if (k <= k_trans && i < QL_NX - 1 && k_trans > 1) {
        const double xi = __ldg(x0 + b * QL_NX + i);
        v = __dadd_rn(xi, __dmul_rn(__ddiv_rn(__dsub_rn(__ldg(xterm + i), xi), (double)(k_trans - 1)), (double)(k - 1)));
    }
    Z[b * ldz + e] = v;
}

// DENSE mode (single evaluations): scatter SPARSE_BLOCK values into the zeroed m x n grid
__global__ void scatter_dense_kernel(const double* __restrict__ vals, const long long* __restrict__ lin,
                                     double* __restrict__ dense, int nnz)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nnz) dense[lin[i]] = vals[i];
}

}  // namespace ql
