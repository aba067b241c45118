// CPU emulation of the matrix-free products (J w, J' y, H v) as the kernels form them, built from the SAME headers
// (layout.h, rk4_dual_gen.h): the generated jvp / vjp / hess_prod routines and the per-knot extra rows in the order
// of eval_prod_kernel (qlnlp_kernels.cuh: prod_pass) and hess_prod_kernel.  tests/test_products_cpu.py checks it bit
// for bit against a left fold of the emulated value streams.  No kinematic rows.  TEST HARNESS ONLY.
#include <cmath>

#include "host_consts.h"
#include "../../quadruped_landing_b200/csrc/layout.h"
#include "../../quadruped_landing_b200/csrc/rk4_dual_gen.h"

static void rk4_jac(const QlClass& c, int k, const double* x, double* jv)
{
    const HostConsts K{c.g, c.mb, c.mf, c.Ib};
    double xn[15];
    if (k >= c.k_trans) ql_rk4_jac_mode3(x, x + 15, K, xn, jv);
    else if (c.init_mode == 1) ql_rk4_jac_mode1(x, x + 15, K, xn, jv);
    else ql_rk4_jac_mode2(x, x + 15, K, xn, jv);
}

static double jtheta_of(const QlClass& c, double th) { return (th > 0) ? (-c.half_lb) * std::cos(th) : c.half_lb * std::cos(th); }

extern "C" {

// out[m_nlp] = J(Z) w
int emul_jvp(int N, int k_trans, int init_mode, double g, double mb, double mf, double lb, const double* Z,
             const double* w, double* out)
{
    QlClass c;
    ql_class_init(&c, N, k_trans, init_mode, g, mb, mf, lb);
    for (int i = 0; i < c.m_nlp; ++i) out[i] = NAN;
    const bool y1 = init_mode == 1;
    for (int k = 1; k <= N; ++k) {
        const double* x = Z + 20 * (k - 1);
        const double* wk = w + 20 * (k - 1);
        const double jt = jtheta_of(c, x[2]);
        if (k == 1) for (int i = 0; i < 15; ++i) out[i] = wk[i];
        if (k == N) for (int i = 0; i < 14; ++i) out[c.c_term + i] = wk[i];
        out[c.c_cfirst + k - 1] = y1 ? wk[4] : wk[6];
        if (k >= k_trans) out[c.c_cother + k - k_trans] = y1 ? wk[6] : wk[4];
        if (k == N - 1) out[c.c_fctrl] = wk[16] + wk[18];
        out[c.c_body + k - 1] = wk[1] + jt * wk[2];
        if (k < N) {
            double jv[QL_NJ_MODE1];
            rk4_jac(c, k, x, jv);
            double* o = out + c.c_dyn + 15 * (k - 1);
            const double* wn = wk + 20;
            const bool jump = k == k_trans - 1;
            if (k >= k_trans) ql_rk4_jvp_mode3(jv, wk, wn, o);
            else if (init_mode == 1) { if (jump) ql_rk4_jvp_mode1_jump(jv, wk, wn, o); else ql_rk4_jvp_mode1(jv, wk, wn, o); }
            else { if (jump) ql_rk4_jvp_mode2_jump(jv, wk, wn, o); else ql_rk4_jvp_mode2(jv, wk, wn, o); }
        }
    }
    return 0;
}

// out[n_nlp] = J(Z)' y
int emul_vjp(int N, int k_trans, int init_mode, double g, double mb, double mf, double lb, const double* Z,
             const double* y, double* out)
{
    QlClass c;
    ql_class_init(&c, N, k_trans, init_mode, g, mb, mf, lb);
    const bool y1 = init_mode == 1;
    for (int k = 1; k <= N; ++k) {
        const double* x = Z + 20 * (k - 1);
        double a[15], o[20];
        for (int j = 0; j < 15; ++j) {
            if (k == 1) a[j] = y[j];
            else {
                const double mi = -y[c.c_dyn + 15 * (k - 2) + j];
                a[j] = (k == N && j < 14) ? y[c.c_term + j] + mi : mi;
            }
        }
        if (k < N) {
            double jv[QL_NJ_MODE1];
            rk4_jac(c, k, x, jv);
            const double* yd = y + c.c_dyn + 15 * (k - 1);
            const bool jump = k == k_trans - 1;
            if (k >= k_trans) ql_rk4_vjp_mode3(jv, yd, a, o);
            else if (init_mode == 1) { if (jump) ql_rk4_vjp_mode1_jump(jv, yd, a, o); else ql_rk4_vjp_mode1(jv, yd, a, o); }
            else { if (jump) ql_rk4_vjp_mode2_jump(jv, yd, a, o); else ql_rk4_vjp_mode2(jv, yd, a, o); }
            if (k == N - 1) { o[16] = o[16] + y[c.c_fctrl]; o[18] = o[18] + y[c.c_fctrl]; }
        } else {
            for (int j = 0; j < 15; ++j) o[j] = a[j];
        }
        const double yf = y[c.c_cfirst + k - 1];
        if (y1) { o[4] = o[4] + yf; if (k >= k_trans) o[6] = o[6] + y[c.c_cother + k - k_trans]; }
        else { o[6] = o[6] + yf; if (k >= k_trans) o[4] = o[4] + y[c.c_cother + k - k_trans]; }
        const double yb = y[c.c_body + k - 1];
        o[1] = o[1] + yb;
        o[2] = o[2] + jtheta_of(c, x[2]) * yb;
        for (int j = 0; j < (k < N ? 20 : 15); ++j) out[20 * (k - 1) + j] = o[j];
    }
    return 0;
}

// out[n_nlp] = H(Z, sigma, lambda) v; cost: knot-major Q[N][15] R[N][5] q[N][15] r[N][5]
int emul_hvp(int N, int k_trans, int init_mode, double g, double mb, double mf, double lb, const double* Q,
             const double* R, const double* q, const double* r, const double* Z, double sigma, const double* lambda,
             const double* v, double* out)
{
    QlClass c;
    ql_class_init(&c, N, k_trans, init_mode, g, mb, mf, lb);
    const HostConsts K{c.g, c.mb, c.mf, c.Ib};
    for (int k = 1; k <= N; ++k) {
        const double* x = Z + 20 * (k - 1);
        const double* u = x + 15;
        const double* vk = v + 20 * (k - 1);
        double* o = out + 20 * (k - 1);
        const double as = c.half_lb * std::sin(x[2]);
        const double tt = lambda[c.c_body + (k - 1)] * ((x[2] > 0) ? as : -as);
        const double* Qk = Q + 15 * (k - 1);
        if (k == N) {
            for (int i = 0; i < 15; ++i) o[i] = ((i == 2) ? sigma * Qk[i] + tt : sigma * Qk[i]) * vk[i];
            continue;
        }
        double lam[15], hv[QL_NH_MODE1], ox[15], ou[4], hx[15], hu[4];
        for (int i = 0; i < 15; ++i) lam[i] = lambda[c.c_dyn + 15 * (k - 1) + i];
        if (k == k_trans - 1) { lam[4] = lam[6] = lam[10] = lam[11] = lam[12] = lam[13] = 0.0; }
        const double h = u[4];
        const double *Rk = R + 5 * (k - 1), *qk = q + 15 * (k - 1), *rk = r + 5 * (k - 1);
        for (int i = 0; i < 15; ++i) { ox[i] = sigma * (h * Qk[i]); hx[i] = sigma * (Qk[i] * x[i] + qk[i]); }
        for (int i = 0; i < 4; ++i) { ou[i] = sigma * (h * Rk[i]); hu[i] = sigma * (Rk[i] * u[i] + rk[i]); }
        const double hh = sigma * (2.0 * (Rk[4] * h + rk[4]) + h * Rk[4]);
        if (k >= k_trans) { ql_rk4_hess_mode3(x, u, K, lam, hv); ql_hess_prod_mode3(hv, ox, ou, hx, hu, hh, tt, vk, o); }
        else if (init_mode == 1) { ql_rk4_hess_mode1(x, u, K, lam, hv); ql_hess_prod_mode1(hv, ox, ou, hx, hu, hh, tt, vk, o); }
        else { ql_rk4_hess_mode2(x, u, K, lam, hv); ql_hess_prod_mode2(hv, ox, ou, hx, hu, hh, tt, vk, o); }
    }
    return 0;
}
}
