// qlnlp_kkt.cuh -- batched solve of the regularised Newton/KKT system of each problem (include/qlnlp.h,
// qlnlp_kkt_solve_batch_device; DESIGN.md section 5, "KKT solve"):
//
//   [ W + diag(sx)   J'       ] [ px ]   [ r1 ]        M = W + diag(sx) + J' diag(dc)^-1 J     (block tridiagonal)
//   [ J             -diag(dc) ] [ pl ] = [ r2 ]        M px = r1 + J' (r2 ./ dc),   pl = (J px - r2) ./ dc
//
// W is block diagonal (one 20x20 block per knot) and every row of J touches one knot, except the dynamics defect of
// step k, which touches knot k (the RK4 block A_k) and knot k+1 (-I on x_(k+1)).  So M's off-diagonal block between
// knots k and k+1 is E_k D_k^-1 A_k, with 15 non-zero rows (D_k, E_k: dc and the -I values of step k's rows).
//
// One warp per problem, knots in sequence.  Knot k's inputs are gathered into a dense local Jacobian G (34 slots x 20
// columns: the rows touching knot k, kkt_slot_row) and the lower triangle of its W block.  Forward sweep:
//   M_kk = W_k + diag(sx_k) + G' D^-1 G - X_(k-1) X_(k-1)'      (X_(k-1) = L_(k,k-1): 15 x 20, previous knot)
//   L_kk = chol(M_kk),  y_k = L_kk^-1 (b_k - X_(k-1) y_(k-1))   (b_k = r1_k + G' (r2 ./ dc))
//   X_k  = E_k D_k^-1 A_k L_kk^-T
// Factor storage: only L_kk (packed lower, 210 doubles) and y_k (20) go to global scratch, 1,840 B per knot; X_k is
// not stored.  The backward sweep gathers knot k again (it needs G for pl anyway) and forms X_k' x_(k+1) as
// L_kk^-1 (A_k' D_k^-1 E_k x_(k+1)):  x_k = L_kk^-T (y_k - X_k' x_(k+1)),  pl = (J px - r2) ./ dc row by row.
//
// The same sweeps split in two (qlnlp_kkt_factor_batch_device, qlnlp_kkt_solve_factored_batch_device):
// kkt_factor_kernel runs the forward sweep without a right-hand side and keeps L_kk and X_k of every knot in the
// caller's factor row (kkt_factor_*), with the J values and dc it read; kkt_solve_factored_kernel forms b_k and y_k from
// that row, keeps y_k in px, and runs the backward sweep.  All three kernels call the per-knot steps below, in the same
// order on the same values, so a factor followed by a factored solve gives the bits of the one-shot solve.
//
// Every value is produced by one lane in a fixed order with explicitly rounded operations, so the bits depend on the
// problem's inputs only (not on B, the batch position, the warp, leading dimensions or alignment).
#pragma once

#include <float.h>

#include "../../include/qlnlp.h"
#include "layout.h"

namespace ql {

constexpr int KKT_SLOTS = 34;          // rows of knot k's local Jacobian (kkt_slot_row)
constexpr int KKT_TRI = QL_NZK * (QL_NZK + 1) / 2;      // packed lower triangle of a 20 x 20 block
constexpr int KKT_FSTRIDE = KKT_TRI + QL_NZK;           // factor scratch per knot: L_kk packed | y_k
constexpr int KKT_XSIZE = QL_NX * QL_NZK;               // X_k = L_(k+1,k): 15 x 20, row-major
constexpr int KKT_FHEAD = 4;                            // factor row header: status | N | k_trans | init_mode

// Layout of a factor row (doubles): the header, L_kk of knots 1..N (KKT_TRI each, packed lower; 120 used at knot N),
// X_k of knots 1..N-1, then the problem's SPARSE_TRUE J values and dc, which the factored solve reads instead of the
// caller's arrays.  The host reports kkt_factor_size through qlnlp_kkt_factor_size.
QL_HD long long kkt_factor_l(const QlClass& c, int k) { (void)c; return KKT_FHEAD + (long long)KKT_TRI * (k - 1); }
QL_HD long long kkt_factor_x(const QlClass& c, int k) { return KKT_FHEAD + (long long)KKT_TRI * c.N + (long long)KKT_XSIZE * (k - 1); }
QL_HD long long kkt_factor_jac(const QlClass& c) { return kkt_factor_x(c, c.N); }
QL_HD long long kkt_factor_dc(const QlClass& c) { return kkt_factor_jac(c) + c.nnz_true; }
QL_HD long long kkt_factor_size(const QlClass& c) { return kkt_factor_dc(c) + c.m_nlp; }

// Constraint row (0-based, g order) held in slot s of knot k's local Jacobian, or -1:
//   0..14   dynamics defect of step k (k < N; A_k) -- at k = N the 14 terminal rows
//   15..29  dynamics defect of step k-1 (-I on x_k) -- at k = 1 the 15 initial-state rows
//   30 contact-first, 31 contact-other (k >= k_trans), 32 final-ctrl (k = N-1), 33 body clearance
// The host maps every SPARSE_TRUE value to its slot with this function (the inverse is not written down twice).
QL_HD int kkt_slot_row(const QlClass& c, int k, int s)
{
    if (s < QL_NX) {
        if (k < c.N) return c.c_dyn + QL_NX * (k - 1) + s;
        return s < QL_NX - 1 ? c.c_term + s : -1;
    }
    if (s < 2 * QL_NX) return k == 1 ? s - QL_NX : c.c_dyn + QL_NX * (k - 2) + (s - QL_NX);
    if (s == 30) return c.c_cfirst + (k - 1);
    if (s == 31) return k >= c.k_trans ? c.c_cother + (k - c.k_trans) : -1;
    if (s == 32) return k == c.N - 1 ? c.c_fctrl : -1;
    return c.c_body + (k - 1);
}

struct KktLaunch {
    QlClass c;
    const unsigned short* jtab;          // [nnz_true]  slot | local column << 8 of every SPARSE_TRUE value
    const unsigned short* htab;          // [nnz_hess]  local row | local column << 8 (row >= column) of every W value
    qlnlp_kkt_io io;
    double* scratch;                     // [gridDim.x][N][KKT_FSTRIDE]: one factor per resident warp
    long long B;
    unsigned* ticket;                    // work counter of the stream (shared with the other kernels' launches)
};

struct KktFactorLaunch {
    QlClass c;
    const unsigned short* jtab;
    const unsigned short* htab;
    qlnlp_kkt_factor_io io;
    long long B;
    unsigned* ticket;
};

struct KktSolveLaunch {
    QlClass c;
    const unsigned short* jtab;
    qlnlp_kkt_rhs_io io;
    long long B;
    unsigned* ticket;
};

struct KktResidualLaunch {
    QlClass c;
    const unsigned short* jtab;
    const unsigned short* htab;
    qlnlp_kkt_residual_io io;
    long long B;
    unsigned* ticket;
};

// The warp's working set of one knot: references to the kernel's own __shared__ arrays (QL_KKT_SHARED).  Declared
// as separate arrays, not as one struct, so that kkt_kernel keeps the shared-memory layout and the register
// allocation it had before the per-knot steps became functions (one struct: 108 registers instead of 168).
struct KktShared {
    double (&G)[KKT_SLOTS][QL_NZK];
    double (&Ms)[QL_NZK][QL_NZK + 1];  // M_kk, then L_kk, lower triangle
    double (&Xs)[QL_NX][QL_NZK + 1];   // X_(k-1), then X_k
    double (&dinv)[KKT_SLOTS];
    double (&dcs)[KKT_SLOTS];
    double (&r2s)[KKT_SLOTS];
    double (&bv)[QL_NZK];
    double (&yv)[QL_NZK];
    double (&xv)[QL_NZK];
    double (&xn)[QL_NZK];
    double (&en)[QL_NX];
};
#define QL_KKT_SHARED(S)                                                                                   \
    __shared__ double G_[KKT_SLOTS][QL_NZK];                                                               \
    __shared__ double Ms_[QL_NZK][QL_NZK + 1];                                                             \
    __shared__ double Xs_[QL_NX][QL_NZK + 1];                                                              \
    __shared__ double dinv_[KKT_SLOTS], dcs_[KKT_SLOTS], r2s_[KKT_SLOTS];                                  \
    __shared__ double bv_[QL_NZK], yv_[QL_NZK], xv_[QL_NZK], xn_[QL_NZK], en_[QL_NX];                      \
    KktShared S{G_, Ms_, Xs_, dinv_, dcs_, r2s_, bv_, yv_, xv_, xn_, en_}

// row a and column b of the packed lower-triangle entry e = a (a + 1) / 2 + b
__device__ __forceinline__ void kkt_tri(int e, int& a, int& b)
{
    a = (int)((__dsqrt_rn(8.0 * e + 1.0) - 1.0) * 0.5);
    while ((a + 1) * (a + 2) / 2 <= e) ++a;
    while (a * (a + 1) / 2 > e) --a;
    b = e - a * (a + 1) / 2;
}

// gather knot k of one problem: G, the per-slot dc, 1/dc, with RHS r2 (and, with W set, the W block into Ms)
template <bool RHS>
__device__ __forceinline__ void kkt_gather(KktShared& S, const QlClass& c, const unsigned short* jtab,
                                           const unsigned short* htab, const double* J, const double* dc,
                                           const double* r2, const double* W, int k, int lane)
{
    for (int i = lane; i < KKT_SLOTS * QL_NZK; i += QL_LANES) (&S.G[0][0])[i] = 0.0;
    if (W) for (int i = lane; i < QL_NZK * (QL_NZK + 1); i += QL_LANES) (&S.Ms[0][0])[i] = 0.0;
    __syncwarp();
    const int j0 = ql_true_run_off(c, k), j1 = k < c.N ? ql_true_run_off(c, k + 1) : c.nnz_true;
    for (int e = j0 + lane; e < j1; e += QL_LANES) {
        const unsigned t = __ldg(jtab + e);
        S.G[t & 0xff][t >> 8] = J[e];
    }
    if (W) {
        const int h0 = ql_hess_run_off(c, k), h1 = h0 + ql_hess_len(c, k);
        for (int e = h0 + lane; e < h1; e += QL_LANES) {
            const unsigned t = __ldg(htab + e);
            S.Ms[t & 0xff][t >> 8] = W[e];
        }
    }
#pragma unroll 1
    for (int s = lane; s < KKT_SLOTS; s += QL_LANES) {      // (34 slots: two lanes take a second one)
        const int r = kkt_slot_row(c, k, s);
        const double d = r >= 0 ? dc[r] : 1.0;
        S.dcs[s] = d;
        S.dinv[s] = r >= 0 ? __drcp_rn(d) : 0.0;
        if (RHS) S.r2s[s] = r >= 0 ? r2[r] : 0.0;
    }
    __syncwarp();
}

// status of a problem's dc: 0, or -1 when an entry is <= 0 or not finite
__device__ __forceinline__ int kkt_dc_status(const QlClass& c, const double* dc, int lane)
{
    bool bad = false;
    for (int i = lane; i < c.m_nlp; i += QL_LANES) {
        const double d = dc[i];
        if (!(d > 0.0 && d <= DBL_MAX)) bad = true;
    }
    return __any_sync(0xffffffffu, bad) ? -1 : 0;
}

// X_(k-1) = E D^-1 A L^-T: apply E, the -I values of knot k's run (k > 1)
__device__ __forceinline__ void kkt_apply_e(KktShared& S, int lane)
{
    if (lane < QL_NX) {
        const double e = S.G[QL_NX + lane][lane];
#pragma unroll 4
        for (int j = 0; j < QL_NZK; ++j) S.Xs[lane][j] = __dmul_rn(e, S.Xs[lane][j]);
    }
}

// M_kk = W_k + diag(sx_k) + G' D^-1 G - X_(k-1) X_(k-1)' (lower triangle, in Ms)
__device__ __forceinline__ void kkt_assemble(KktShared& S, const double* sx, int k, int nk, int z0, int lane)
{
    for (int e = lane; e < nk * (nk + 1) / 2; e += QL_LANES) {
        int a, bb;
        kkt_tri(e, a, bb);
        double m = S.Ms[a][bb];
        if (a == bb && sx) m = __dadd_rn(m, sx[z0 + a]);
        double acc = 0.0;
        for (int s = 0; s < KKT_SLOTS; ++s) acc = __fma_rn(__dmul_rn(S.G[s][a], S.dinv[s]), S.G[s][bb], acc);
        m = __dadd_rn(m, acc);
        if (k > 1 && a < QL_NX) {
            double u = 0.0;
            for (int j = 0; j < QL_NZK; ++j) u = __fma_rn(S.Xs[a][j], S.Xs[bb][j], u);
            m = __dsub_rn(m, u);
        }
        S.Ms[a][bb] = m;
    }
}

// b_k - X_(k-1) y_(k-1) into bv (b_k = r1_k + G' (r2 ./ dc))
__device__ __forceinline__ void kkt_form_b(KktShared& S, const double* r1, int k, int nk, int z0, int lane)
{
    if (lane < nk) {
        double acc = 0.0;
        for (int s = 0; s < KKT_SLOTS; ++s) acc = __fma_rn(S.G[s][lane], __ddiv_rn(S.r2s[s], S.dcs[s]), acc);
        double v = __dadd_rn(r1[z0 + lane], acc);
        if (k > 1 && lane < QL_NX) {
            double u = 0.0;
            for (int j = 0; j < QL_NZK; ++j) u = __fma_rn(S.Xs[lane][j], S.yv[j], u);
            v = __dsub_rn(v, u);
        }
        S.bv[lane] = v;
    }
}

// Cholesky of M_kk in place (lane i owns row i); a pivot that is not a finite positive number sets status = k.
// (status as an argument, not a returned flag: kkt_kernel then keeps its register allocation.)
__device__ __forceinline__ void kkt_cholesky(KktShared& S, int nk, int k, int& status, int lane)
{
    for (int j = 0; j < nk; ++j) {
        __syncwarp();
        const double d = S.Ms[j][j];
        if (!(d > 0.0 && d <= DBL_MAX)) { status = k; break; }
        const double ljj = __dsqrt_rn(d);
        __syncwarp();
        if (lane == j) S.Ms[j][j] = ljj;
        if (lane > j && lane < nk) S.Ms[lane][j] = __ddiv_rn(S.Ms[lane][j], ljj);
        __syncwarp();
        if (lane > j && lane < nk)
            for (int q = j + 1; q <= lane; ++q) S.Ms[lane][q] = __fma_rn(-S.Ms[lane][j], S.Ms[q][j], S.Ms[lane][q]);
    }
}

// out = L^-1 w (w is overwritten), L = Ms, order nk
__device__ __forceinline__ void kkt_lsolve(KktShared& S, double* w, double* out, int nk, int lane)
{
    for (int j = 0; j < nk; ++j) {
        __syncwarp();
        const double yj = __ddiv_rn(w[j], S.Ms[j][j]);
        if (lane == j) out[j] = yj;
        if (lane > j && lane < nk) w[lane] = __fma_rn(-S.Ms[lane][j], yj, w[lane]);
    }
    __syncwarp();
}

// out = L^-T r (r is overwritten)
__device__ __forceinline__ void kkt_ltsolve(KktShared& S, double* r, double* out, int nk, int lane)
{
    for (int j = nk - 1; j >= 0; --j) {
        __syncwarp();
        const double xj = __ddiv_rn(r[j], S.Ms[j][j]);
        if (lane == j) out[j] = xj;
        if (lane < j) r[lane] = __fma_rn(-S.Ms[j][lane], xj, r[lane]);
    }
    __syncwarp();
}

// X_k without E: rows of D^-1 A_k L_kk^-T, one lane per row (k < N)
__device__ __forceinline__ void kkt_form_x(KktShared& S, int lane)
{
    if (lane < QL_NX) {
        const double di = S.dinv[lane];
        for (int j = 0; j < QL_NZK; ++j) {
            double s = __dmul_rn(di, S.G[lane][j]);
            for (int q = 0; q < j; ++q) s = __fma_rn(-S.Ms[j][q], S.Xs[lane][q], s);
            S.Xs[lane][j] = __ddiv_rn(s, S.Ms[j][j]);
        }
    }
}

// packed L_kk between Ms and global memory
__device__ __forceinline__ void kkt_store_l(KktShared& S, double* f, int nk, int lane)
{
    for (int e = lane; e < nk * (nk + 1) / 2; e += QL_LANES) {
        int a, bb;
        kkt_tri(e, a, bb);
        f[e] = S.Ms[a][bb];
    }
}

__device__ __forceinline__ void kkt_load_l(KktShared& S, const double* f, int nk, int lane)
{
    for (int e = lane; e < nk * (nk + 1) / 2; e += QL_LANES) {
        int a, bb;
        kkt_tri(e, a, bb);
        S.Ms[a][bb] = f[e];
    }
}

// Backward step at knot k, with knot k gathered, L_kk in Ms and y_k in bv: x_k into px, the pl rows that close at
// knot k, and E_k, x_k kept for knot k-1.
__device__ __forceinline__ void kkt_backward(KktShared& S, const QlClass& c, int k, int nk, int z0, double* px,
                                             double* pl, int lane)
{
    if (k < c.N && lane < QL_NZK) {       // v = A_k' D^-1 E x_(k+1)
        double v = 0.0;
        for (int i = 0; i < QL_NX; ++i) v = __fma_rn(S.G[i][lane], __dmul_rn(__dmul_rn(S.en[i], S.dinv[i]), S.xn[i]), v);
        S.yv[lane] = v;
    }
    __syncwarp();
    if (k < c.N) {
        kkt_lsolve(S, S.yv, S.xv, QL_NZK, lane);   // X_k' x_(k+1) = L_kk^-1 v
        if (lane < QL_NZK) S.bv[lane] = __dsub_rn(S.bv[lane], S.xv[lane]);
    }
    kkt_ltsolve(S, S.bv, S.xv, nk, lane);
    if (lane < nk) px[z0 + lane] = S.xv[lane];
#pragma unroll 1
    for (int s = lane; s < KKT_SLOTS; s += QL_LANES) {
        const int r = (s < QL_NX || s >= 2 * QL_NX || k == 1) ? kkt_slot_row(c, k, s) : -1;
        if (r >= 0) {
            double acc = 0.0;
            for (int j = 0; j < nk; ++j) acc = __fma_rn(S.G[s][j], S.xv[j], acc);
            if (s < QL_NX && k < c.N) acc = __fma_rn(S.en[s], S.xn[s], acc);
            pl[r] = __ddiv_rn(__dsub_rn(acc, S.r2s[s]), S.dcs[s]);
        }
    }
    __syncwarp();
    if (lane < QL_NX) S.en[lane] = S.G[QL_NX + lane][lane];
    if (lane < QL_NZK) S.xn[lane] = S.xv[lane];
    __syncwarp();
}

// px and pl of a problem with a non-zero status
__device__ __forceinline__ void kkt_fill_nan(const QlClass& c, double* px, double* pl, int lane)
{
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    for (int i = lane; i < c.n_nlp; i += QL_LANES) px[i] = nan;
    for (int i = lane; i < c.m_nlp; i += QL_LANES) pl[i] = nan;
}

// the last CTA to leave re-arms the counters for the next launch on this stream
__device__ __forceinline__ void kkt_rearm(unsigned* ticket, int lane)
{
    if (lane == 0) {
        __threadfence();
        if (atomicAdd(ticket + 1, 1u) == gridDim.x - 1) {
            ticket[0] = 0u;
            ticket[1] = 0u;
        }
    }
}

__global__ void __launch_bounds__(QL_LANES, 8) kkt_kernel(const __grid_constant__ KktLaunch P)
{
    QL_KKT_SHARED(S);
    const QlClass& c = P.c;
    const int lane = threadIdx.x;
    const unsigned full = 0xffffffffu;
    double* const fac = P.scratch + (long long)blockIdx.x * c.N * KKT_FSTRIDE;

    auto take_issue = [&]() -> unsigned { return lane == 0 ? atomicAdd(P.ticket, 1u) : 0u; };
    auto take_get = [&](unsigned t) -> long long { return (long long)__shfl_sync(full, t, 0); };
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");     // (a predecessor launched with the dependent-launch attribute)
    long long b = take_get(take_issue());
    while (b < P.B) {
        const unsigned tkt = take_issue();
        const double* const W = P.io.hess + b * P.io.ldhess;
        const double* const J = P.io.jac + b * P.io.ldjac;
        const double* const sx = P.io.sx ? P.io.sx + b * P.io.ldsx : nullptr;
        const double* const dc = P.io.dc + b * P.io.lddc;
        const double* const r1 = P.io.r1 + b * P.io.ldr1;
        const double* const r2 = P.io.r2 + b * P.io.ldr2;
        double* const px = P.io.px + b * P.io.ldpx;
        double* const pl = P.io.pl + b * P.io.ldpl;

        int status = kkt_dc_status(c, dc, lane);

        // ---- forward sweep: factor and forward substitution, knot by knot
        for (int k = 1; status == 0 && k <= c.N; ++k) {
            const int nk = k < c.N ? QL_NZK : QL_NX;
            const int z0 = QL_NZK * (k - 1);
            kkt_gather<true>(S, c, P.jtab, P.htab, J, dc, r2, W, k, lane);
            if (k > 1) kkt_apply_e(S, lane);
            __syncwarp();
            kkt_assemble(S, sx, k, nk, z0, lane);
            kkt_form_b(S, r1, k, nk, z0, lane);
            kkt_cholesky(S, nk, k, status, lane);
            if (status) break;
            kkt_lsolve(S, S.bv, S.yv, nk, lane);
            double* const fk = fac + (long long)(k - 1) * KKT_FSTRIDE;
            kkt_store_l(S, fk, nk, lane);
            if (lane < nk) fk[KKT_TRI + lane] = S.yv[lane];
            if (k < c.N) kkt_form_x(S, lane);
            __syncwarp();
        }

        // ---- backward sweep: x_k from knot N down, pl of the rows finished at knot k
        for (int k = c.N; status == 0 && k >= 1; --k) {
            const int nk = k < c.N ? QL_NZK : QL_NX;
            const int z0 = QL_NZK * (k - 1);
            kkt_gather<true>(S, c, P.jtab, P.htab, J, dc, r2, nullptr, k, lane);
            const double* const fk = fac + (long long)(k - 1) * KKT_FSTRIDE;
            kkt_load_l(S, fk, nk, lane);
            if (lane < nk) S.bv[lane] = fk[KKT_TRI + lane];
            kkt_backward(S, c, k, nk, z0, px, pl, lane);
        }
        if (status != 0) kkt_fill_nan(c, px, pl, lane);
        if (lane == 0) P.io.status[b] = status;
        __syncwarp();
        b = take_get(tkt);
    }
    kkt_rearm(P.ticket, lane);
}

// Forward sweep without a right-hand side: L_kk and X_k (E applied) of every knot into the problem's factor row, with
// the J values and dc the sweep read, the status and the class stamp.
__global__ void __launch_bounds__(QL_LANES, 8) kkt_factor_kernel(const __grid_constant__ KktFactorLaunch P)
{
    QL_KKT_SHARED(S);
    const QlClass& c = P.c;
    const int lane = threadIdx.x;
    const unsigned full = 0xffffffffu;

    auto take_issue = [&]() -> unsigned { return lane == 0 ? atomicAdd(P.ticket, 1u) : 0u; };
    auto take_get = [&](unsigned t) -> long long { return (long long)__shfl_sync(full, t, 0); };
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
    long long b = take_get(take_issue());
    while (b < P.B) {
        const unsigned tkt = take_issue();
        const double* const W = P.io.hess + b * P.io.ldhess;
        const double* const J = P.io.jac + b * P.io.ldjac;
        const double* const sx = P.io.sx ? P.io.sx + b * P.io.ldsx : nullptr;
        const double* const dc = P.io.dc + b * P.io.lddc;
        double* const F = P.io.factor + b * P.io.ldfactor;

        double* const Fj = F + kkt_factor_jac(c);
        double* const Fd = F + kkt_factor_dc(c);
        for (int e = lane; e < c.nnz_true; e += QL_LANES) Fj[e] = J[e];
        for (int i = lane; i < c.m_nlp; i += QL_LANES) Fd[i] = dc[i];
        int status = kkt_dc_status(c, dc, lane);

        for (int k = 1; status == 0 && k <= c.N; ++k) {
            const int nk = k < c.N ? QL_NZK : QL_NX;
            const int z0 = QL_NZK * (k - 1);
            kkt_gather<false>(S, c, P.jtab, P.htab, J, dc, nullptr, W, k, lane);
            if (k > 1) kkt_apply_e(S, lane);
            __syncwarp();
            if (k > 1) {
                double* const fx = F + kkt_factor_x(c, k - 1);
                for (int e = lane; e < KKT_XSIZE; e += QL_LANES) fx[e] = S.Xs[e / QL_NZK][e % QL_NZK];
            }
            kkt_assemble(S, sx, k, nk, z0, lane);
            kkt_cholesky(S, nk, k, status, lane);
            if (status) break;
            __syncwarp();
            double* const fl = F + kkt_factor_l(c, k);
            kkt_store_l(S, fl, nk, lane);
            for (int e = nk * (nk + 1) / 2 + lane; e < KKT_TRI; e += QL_LANES) fl[e] = 0.0;   // knot N: the unused tail
            if (k < c.N) kkt_form_x(S, lane);
            __syncwarp();
        }
        if (lane == 0) {
            F[0] = (double)status;
            F[1] = (double)c.N;
            F[2] = (double)c.k_trans;
            F[3] = (double)c.init_mode;
            P.io.status[b] = status;
        }
        __syncwarp();
        b = take_get(tkt);
    }
    kkt_rearm(P.ticket, lane);
}

// One right-hand side per warp against a kept factor: forward substitution (y_k kept in px), then the backward sweep.
__global__ void __launch_bounds__(QL_LANES, 8) kkt_solve_factored_kernel(const __grid_constant__ KktSolveLaunch P)
{
    QL_KKT_SHARED(S);
    const QlClass& c = P.c;
    const int lane = threadIdx.x;
    const unsigned full = 0xffffffffu;

    auto take_issue = [&]() -> unsigned { return lane == 0 ? atomicAdd(P.ticket, 1u) : 0u; };
    auto take_get = [&](unsigned t) -> long long { return (long long)__shfl_sync(full, t, 0); };
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
    long long b = take_get(take_issue());
    while (b < P.B) {
        const unsigned tkt = take_issue();
        const double* const r1 = P.io.r1 + b * P.io.ldr1;
        const double* const r2 = P.io.r2 + b * P.io.ldr2;
        double* const px = P.io.px + b * P.io.ldpx;
        double* const pl = P.io.pl + b * P.io.ldpl;
        const long long f = P.io.index ? P.io.index[b] : b;
        const double* F = P.io.factor;
        int status = -2;
        if (f >= 0 && f < P.io.nfactor) {
            F += f * P.io.ldfactor;
            const bool same = F[1] == (double)c.N && F[2] == (double)c.k_trans && F[3] == (double)c.init_mode;
            status = same ? (int)F[0] : -3;
        }
        const double* const J = F + kkt_factor_jac(c);
        const double* const dc = F + kkt_factor_dc(c);

        // ---- forward substitution: y_k = L_kk^-1 (b_k - X_(k-1) y_(k-1)), kept in px until the backward sweep
        for (int k = 1; status == 0 && k <= c.N; ++k) {
            const int nk = k < c.N ? QL_NZK : QL_NX;
            const int z0 = QL_NZK * (k - 1);
            kkt_gather<true>(S, c, P.jtab, nullptr, J, dc, r2, nullptr, k, lane);
            if (k > 1) {
                const double* const fx = F + kkt_factor_x(c, k - 1);
                for (int e = lane; e < KKT_XSIZE; e += QL_LANES) S.Xs[e / QL_NZK][e % QL_NZK] = fx[e];
            }
            kkt_load_l(S, F + kkt_factor_l(c, k), nk, lane);
            __syncwarp();
            kkt_form_b(S, r1, k, nk, z0, lane);
            kkt_lsolve(S, S.bv, S.yv, nk, lane);
            if (lane < nk) px[z0 + lane] = S.yv[lane];
        }

        // ---- backward sweep, as in kkt_kernel
        for (int k = c.N; status == 0 && k >= 1; --k) {
            const int nk = k < c.N ? QL_NZK : QL_NX;
            const int z0 = QL_NZK * (k - 1);
            kkt_gather<true>(S, c, P.jtab, nullptr, J, dc, r2, nullptr, k, lane);
            kkt_load_l(S, F + kkt_factor_l(c, k), nk, lane);
            if (lane < nk) S.bv[lane] = px[z0 + lane];
            kkt_backward(S, c, k, nk, z0, px, pl, lane);
        }
        if (status != 0) kkt_fill_nan(c, px, pl, lane);
        if (lane == 0) P.io.status[b] = status;
        __syncwarp();
        b = take_get(tkt);
    }
    kkt_rearm(P.ticket, lane);
}

// Residual of the system a solve was asked for, with the matrix the solve read (qlnlp_kkt_residual_batch_device):
//   s1 = r1 - (W + diag(sx)) px - J' pl,   s2 = r2 - J px + dc .* pl.
// Knots from N down to 1, as the backward sweep: knot k's G and W block gathered (with pl in place of r2, so r2s holds
// pl of each slot), lane a folds s1 of knot k's variable a, and the rows that close at knot k (kkt_backward's) fold s2,
// a defect row of step k taking the -I of knot k+1 from en, kept from the previous knot.  Each entry is a left fold of
// fused multiply-adds from r, in the order include/qlnlp.h states; W_aa + sx_a is rounded once first, as K holds it.
__global__ void __launch_bounds__(QL_LANES, 8) kkt_residual_kernel(const __grid_constant__ KktResidualLaunch P)
{
    QL_KKT_SHARED(S);
    const QlClass& c = P.c;
    const int lane = threadIdx.x;
    const unsigned full = 0xffffffffu;

    auto take_issue = [&]() -> unsigned { return lane == 0 ? atomicAdd(P.ticket, 1u) : 0u; };
    auto take_get = [&](unsigned t) -> long long { return (long long)__shfl_sync(full, t, 0); };
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
    long long b = take_get(take_issue());
    while (b < P.B) {
        const unsigned tkt = take_issue();
        const double* const W = P.io.hess + b * P.io.ldhess;
        const double* const J = P.io.jac + b * P.io.ldjac;
        const double* const sx = P.io.sx ? P.io.sx + b * P.io.ldsx : nullptr;
        const double* const dc = P.io.dc + b * P.io.lddc;
        const double* const r1 = P.io.r1 + b * P.io.ldr1;
        const double* const r2 = P.io.r2 + b * P.io.ldr2;
        const double* const px = P.io.px + b * P.io.ldpx;
        const double* const pl = P.io.pl + b * P.io.ldpl;
        double* const s1 = P.io.s1 + b * P.io.lds1;
        double* const s2 = P.io.s2 + b * P.io.lds2;

        for (int k = c.N; k >= 1; --k) {
            const int nk = k < c.N ? QL_NZK : QL_NX;
            const int z0 = QL_NZK * (k - 1);
            kkt_gather<true>(S, c, P.jtab, P.htab, J, dc, pl, W, k, lane);
            if (lane < nk) S.xv[lane] = px[z0 + lane];
            __syncwarp();
            if (lane < nk) {               // s1: W row (mirrored, diagonal with sx), then J' column, slot by slot
                double acc = r1[z0 + lane];
                for (int j = 0; j < nk; ++j) {
                    double w = j <= lane ? S.Ms[lane][j] : S.Ms[j][lane];
                    if (j == lane && sx) w = __dadd_rn(w, sx[z0 + j]);
                    acc = __fma_rn(-w, S.xv[j], acc);
                }
                for (int s = 0; s < KKT_SLOTS; ++s) acc = __fma_rn(-S.G[s][lane], S.r2s[s], acc);
                s1[z0 + lane] = acc;
            }
#pragma unroll 1
            for (int s = lane; s < KKT_SLOTS; s += QL_LANES) {     // s2: knot k's columns, the -I of knot k+1, dc pl
                const int r = (s < QL_NX || s >= 2 * QL_NX || k == 1) ? kkt_slot_row(c, k, s) : -1;
                if (r >= 0) {
                    double acc = r2[r];
                    for (int j = 0; j < nk; ++j) acc = __fma_rn(-S.G[s][j], S.xv[j], acc);
                    if (s < QL_NX && k < c.N) acc = __fma_rn(-S.en[s], px[z0 + QL_NZK + s], acc);
                    s2[r] = __fma_rn(S.dcs[s], S.r2s[s], acc);
                }
            }
            __syncwarp();
            if (lane < QL_NX) S.en[lane] = S.G[QL_NX + lane][lane];
            __syncwarp();
        }
        b = take_get(tkt);
    }
    kkt_rearm(P.ticket, lane);
}

}  // namespace ql
