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
// Every value is produced by one lane in a fixed order with explicitly rounded operations, so the bits depend on the
// problem's inputs only (not on B, the batch position, the warp, leading dimensions or alignment).
#pragma once

#include <float.h>

#include "layout.h"

namespace ql {

constexpr int KKT_SLOTS = 34;          // rows of knot k's local Jacobian (kkt_slot_row)
constexpr int KKT_TRI = QL_NZK * (QL_NZK + 1) / 2;      // packed lower triangle of a 20 x 20 block
constexpr int KKT_FSTRIDE = KKT_TRI + QL_NZK;           // factor scratch per knot: L_kk packed | y_k

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
    const double* hess; long long ldhess;
    const double* jac; long long ldjac;
    const double* sx; long long ldsx;    // or nullptr: 0
    const double* dc; long long lddc;
    const double* r1; long long ldr1;
    const double* r2; long long ldr2;
    double* px; long long ldpx;
    double* pl; long long ldpl;
    int* status;
    double* scratch;                     // [gridDim.x][N][KKT_FSTRIDE]: one factor per resident warp
    long long B;
    unsigned* ticket;                    // work counter of the stream (shared with the other kernels' launches)
};

// row a and column b of the packed lower-triangle entry e = a (a + 1) / 2 + b
__device__ __forceinline__ void kkt_tri(int e, int& a, int& b)
{
    a = (int)((__dsqrt_rn(8.0 * e + 1.0) - 1.0) * 0.5);
    while ((a + 1) * (a + 2) / 2 <= e) ++a;
    while (a * (a + 1) / 2 > e) --a;
    b = e - a * (a + 1) / 2;
}

__global__ void __launch_bounds__(QL_LANES, 8) kkt_kernel(const __grid_constant__ KktLaunch P)
{
    __shared__ double G[KKT_SLOTS][QL_NZK];
    __shared__ double Ms[QL_NZK][QL_NZK + 1];     // M_kk, then L_kk, lower triangle
    __shared__ double Xs[QL_NX][QL_NZK + 1];      // X_(k-1), then X_k
    __shared__ double dinv[KKT_SLOTS], dcs[KKT_SLOTS], r2s[KKT_SLOTS];
    __shared__ double bv[QL_NZK], yv[QL_NZK], xv[QL_NZK], xn[QL_NZK], en[QL_NX];
    const QlClass& c = P.c;
    const int lane = threadIdx.x;
    const unsigned full = 0xffffffffu;
    double* const fac = P.scratch + (long long)blockIdx.x * c.N * KKT_FSTRIDE;

    // gather knot k of problem b: G, the per-slot dc, 1/dc, r2 (and, with W set, the W block into Ms)
    auto gather = [&](const double* J, const double* dc, const double* r2, const double* W, int k) {
        for (int i = lane; i < KKT_SLOTS * QL_NZK; i += QL_LANES) (&G[0][0])[i] = 0.0;
        if (W) for (int i = lane; i < QL_NZK * (QL_NZK + 1); i += QL_LANES) (&Ms[0][0])[i] = 0.0;
        __syncwarp();
        const int j0 = ql_true_run_off(c, k), j1 = k < c.N ? ql_true_run_off(c, k + 1) : c.nnz_true;
        for (int e = j0 + lane; e < j1; e += QL_LANES) {
            const unsigned t = __ldg(P.jtab + e);
            G[t & 0xff][t >> 8] = J[e];
        }
        if (W) {
            const int h0 = ql_hess_run_off(c, k), h1 = h0 + ql_hess_len(c, k);
            for (int e = h0 + lane; e < h1; e += QL_LANES) {
                const unsigned t = __ldg(P.htab + e);
                Ms[t & 0xff][t >> 8] = W[e];
            }
        }
#pragma unroll 1
        for (int s = lane; s < KKT_SLOTS; s += QL_LANES) {      // (34 slots: two lanes take a second one)
            const int r = kkt_slot_row(c, k, s);
            const double d = r >= 0 ? dc[r] : 1.0;
            dcs[s] = d;
            dinv[s] = r >= 0 ? __drcp_rn(d) : 0.0;
            r2s[s] = r >= 0 ? r2[r] : 0.0;
        }
        __syncwarp();
    };
    // out = L^-1 w (w is overwritten), L = Ms, order nk
    auto lsolve = [&](double* w, double* out, int nk) {
        for (int j = 0; j < nk; ++j) {
            __syncwarp();
            const double yj = __ddiv_rn(w[j], Ms[j][j]);
            if (lane == j) out[j] = yj;
            if (lane > j && lane < nk) w[lane] = __fma_rn(-Ms[lane][j], yj, w[lane]);
        }
        __syncwarp();
    };
    // out = L^-T r (r is overwritten)
    auto ltsolve = [&](double* r, double* out, int nk) {
        for (int j = nk - 1; j >= 0; --j) {
            __syncwarp();
            const double xj = __ddiv_rn(r[j], Ms[j][j]);
            if (lane == j) out[j] = xj;
            if (lane < j) r[lane] = __fma_rn(-Ms[j][lane], xj, r[lane]);
        }
        __syncwarp();
    };

    auto take_issue = [&]() -> unsigned { return lane == 0 ? atomicAdd(P.ticket, 1u) : 0u; };
    auto take_get = [&](unsigned t) -> long long { return (long long)__shfl_sync(full, t, 0); };
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");     // (a predecessor launched with the dependent-launch attribute)
    long long b = take_get(take_issue());
    while (b < P.B) {
        const unsigned tkt = take_issue();
        const double* const W = P.hess + b * P.ldhess;
        const double* const J = P.jac + b * P.ldjac;
        const double* const sx = P.sx ? P.sx + b * P.ldsx : nullptr;
        const double* const dc = P.dc + b * P.lddc;
        const double* const r1 = P.r1 + b * P.ldr1;
        const double* const r2 = P.r2 + b * P.ldr2;
        double* const px = P.px + b * P.ldpx;
        double* const pl = P.pl + b * P.ldpl;

        bool bad = false;
        for (int i = lane; i < c.m_nlp; i += QL_LANES) {
            const double d = dc[i];
            if (!(d > 0.0 && d <= DBL_MAX)) bad = true;
        }
        int status = __any_sync(full, bad) ? -1 : 0;

        // ---- forward sweep: factor and forward substitution, knot by knot
        for (int k = 1; status == 0 && k <= c.N; ++k) {
            const int nk = k < c.N ? QL_NZK : QL_NX;
            const int z0 = QL_NZK * (k - 1);
            gather(J, dc, r2, W, k);
            if (k > 1 && lane < QL_NX) {          // X_(k-1) = E D^-1 A L^-T: apply E, the -I values of knot k's run
                const double e = G[QL_NX + lane][lane];
#pragma unroll 4
                for (int j = 0; j < QL_NZK; ++j) Xs[lane][j] = __dmul_rn(e, Xs[lane][j]);
            }
            __syncwarp();
            for (int e = lane; e < nk * (nk + 1) / 2; e += QL_LANES) {
                int a, bb;
                kkt_tri(e, a, bb);
                double m = Ms[a][bb];
                if (a == bb && sx) m = __dadd_rn(m, sx[z0 + a]);
                double acc = 0.0;
                for (int s = 0; s < KKT_SLOTS; ++s) acc = __fma_rn(__dmul_rn(G[s][a], dinv[s]), G[s][bb], acc);
                m = __dadd_rn(m, acc);
                if (k > 1 && a < QL_NX) {
                    double u = 0.0;
                    for (int j = 0; j < QL_NZK; ++j) u = __fma_rn(Xs[a][j], Xs[bb][j], u);
                    m = __dsub_rn(m, u);
                }
                Ms[a][bb] = m;
            }
            if (lane < nk) {
                double acc = 0.0;
                for (int s = 0; s < KKT_SLOTS; ++s) acc = __fma_rn(G[s][lane], __ddiv_rn(r2s[s], dcs[s]), acc);
                double v = __dadd_rn(r1[z0 + lane], acc);
                if (k > 1 && lane < QL_NX) {
                    double u = 0.0;
                    for (int j = 0; j < QL_NZK; ++j) u = __fma_rn(Xs[lane][j], yv[j], u);
                    v = __dsub_rn(v, u);
                }
                bv[lane] = v;
            }
            // Cholesky of M_kk in place (lane i owns row i); a pivot that is not a finite positive number stops the sweep
            for (int j = 0; j < nk; ++j) {
                __syncwarp();
                const double d = Ms[j][j];
                if (!(d > 0.0 && d <= DBL_MAX)) { status = k; break; }
                const double ljj = __dsqrt_rn(d);
                __syncwarp();
                if (lane == j) Ms[j][j] = ljj;
                if (lane > j && lane < nk) Ms[lane][j] = __ddiv_rn(Ms[lane][j], ljj);
                __syncwarp();
                if (lane > j && lane < nk)
                    for (int q = j + 1; q <= lane; ++q) Ms[lane][q] = __fma_rn(-Ms[lane][j], Ms[q][j], Ms[lane][q]);
            }
            if (status) break;
            lsolve(bv, yv, nk);
            double* const fk = fac + (long long)(k - 1) * KKT_FSTRIDE;
            for (int e = lane; e < nk * (nk + 1) / 2; e += QL_LANES) {
                int a, bb;
                kkt_tri(e, a, bb);
                fk[e] = Ms[a][bb];
            }
            if (lane < nk) fk[KKT_TRI + lane] = yv[lane];
            if (k < c.N && lane < QL_NX) {        // X_k without E: rows of D^-1 A_k L_kk^-T, one lane per row
                const double di = dinv[lane];
                for (int j = 0; j < QL_NZK; ++j) {
                    double s = __dmul_rn(di, G[lane][j]);
                    for (int q = 0; q < j; ++q) s = __fma_rn(-Ms[j][q], Xs[lane][q], s);
                    Xs[lane][j] = __ddiv_rn(s, Ms[j][j]);
                }
            }
            __syncwarp();
        }

        // ---- backward sweep: x_k from knot N down, pl of the rows finished at knot k
        for (int k = c.N; status == 0 && k >= 1; --k) {
            const int nk = k < c.N ? QL_NZK : QL_NX;
            const int z0 = QL_NZK * (k - 1);
            gather(J, dc, r2, nullptr, k);
            const double* const fk = fac + (long long)(k - 1) * KKT_FSTRIDE;
            for (int e = lane; e < nk * (nk + 1) / 2; e += QL_LANES) {
                int a, bb;
                kkt_tri(e, a, bb);
                Ms[a][bb] = fk[e];
            }
            if (lane < nk) bv[lane] = fk[KKT_TRI + lane];
            if (k < c.N && lane < QL_NZK) {       // v = A_k' D^-1 E x_(k+1)
                double v = 0.0;
                for (int i = 0; i < QL_NX; ++i) v = __fma_rn(G[i][lane], __dmul_rn(__dmul_rn(en[i], dinv[i]), xn[i]), v);
                yv[lane] = v;
            }
            __syncwarp();
            if (k < c.N) {
                lsolve(yv, xv, QL_NZK);           // X_k' x_(k+1) = L_kk^-1 v
                if (lane < QL_NZK) bv[lane] = __dsub_rn(bv[lane], xv[lane]);
            }
            ltsolve(bv, xv, nk);
            if (lane < nk) px[z0 + lane] = xv[lane];
#pragma unroll 1
            for (int s = lane; s < KKT_SLOTS; s += QL_LANES) {
                const int r = (s < QL_NX || s >= 2 * QL_NX || k == 1) ? kkt_slot_row(c, k, s) : -1;
                if (r >= 0) {
                    double acc = 0.0;
                    for (int j = 0; j < nk; ++j) acc = __fma_rn(G[s][j], xv[j], acc);
                    if (s < QL_NX && k < c.N) acc = __fma_rn(en[s], xn[s], acc);
                    pl[r] = __ddiv_rn(__dsub_rn(acc, r2s[s]), dcs[s]);
                }
            }
            __syncwarp();
            if (lane < QL_NX) en[lane] = G[QL_NX + lane][lane];
            if (lane < QL_NZK) xn[lane] = xv[lane];
            __syncwarp();
        }
        if (status != 0) {
            const double nan = __longlong_as_double(0x7ff8000000000000LL);
            for (int i = lane; i < c.n_nlp; i += QL_LANES) px[i] = nan;
            for (int i = lane; i < c.m_nlp; i += QL_LANES) pl[i] = nan;
        }
        if (lane == 0) P.status[b] = status;
        __syncwarp();
        b = take_get(tkt);
    }
    // the last CTA to leave re-arms the counters for the next launch on this stream
    if (lane == 0) {
        __threadfence();
        if (atomicAdd(P.ticket + 1, 1u) == gridDim.x - 1) {
            P.ticket[0] = 0u;
            P.ticket[1] = 0u;
        }
    }
}

}  // namespace ql
