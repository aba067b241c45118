// Host twin of the generated device code (quadruped_landing_b200/csrc/rk4_dual_gen.h), used by
// tests/test_rk4_gen.py to check -- on the CPU, bit for bit -- that the sparsity-exploiting
// straight-line code equals the oracle's dense 20-wide dual evaluation.
// Build: g++ -O2 -ffp-contract=off -fPIC -shared (done by the test).
#include <cstring>

#include <cmath>
#include "host_consts.h"
#include "../../quadruped_landing_b200/csrc/fastdiv.h"
#include "../../quadruped_landing_b200/csrc/rk4_dual_gen.h"

extern "C" {

// xn[15], J[15*20] column-major (J[i + 15*j]); entries outside the pattern are set to 0.
void host_rk4_jac(int mode, const double* x, const double* u, double g, double mb, double mf, double lb,
                  double* xn, double* J)
{
    const HostConsts K{g, mb, mf, mb * (lb * lb) / 12};
    double jv[QL_NJ_MODE1 > QL_NJ_MODE3 ? QL_NJ_MODE1 : QL_NJ_MODE3];
    std::memset(J, 0, sizeof(double) * 300);
#define SCATTER(M)                                                                                         \
    ql_rk4_jac_mode##M(x, u, K, xn, jv);                                                                   \
    for (int n = 0; n < QL_NJ_MODE##M; ++n) J[QL_PAT_I_MODE##M[n] + 15 * QL_PAT_J_MODE##M[n]] = jv[n];       \
    for (int n = 0; n < QL_NJC_MODE##M; ++n) J[QL_CPAT_I_MODE##M[n] + 15 * QL_CPAT_J_MODE##M[n]] = QL_CPAT_V_MODE##M[n];
    if (mode == 1) { SCATTER(1) } else if (mode == 2) { SCATTER(2) } else { SCATTER(3) }
#undef SCATTER
}

void host_rk4(int mode, const double* x, const double* u, double g, double mb, double mf, double lb, double* xn)
{
    const HostConsts K{g, mb, mf, mb * (lb * lb) / 12};
    if (mode == 1) ql_rk4_mode1(x, u, K, xn);
    else if (mode == 2) ql_rk4_mode2(x, u, K, xn);
    else ql_rk4_mode3(x, u, K, xn);
}

// The kernels divide by the model constants with csrc/fastdiv.h.  Sweeps per_binade numerators of each binade of the
// double range plus the special values: returns how many inside the formula's domain give bits different from the IEEE
// quotient a / b, and counts those outside it, and those of them that break the documented behaviour there.
long long host_count_fastdiv_mismatches(double b, int per_binade, unsigned long long seed, long long* outside,
                                        long long* outside_bad)
{
    return ql::fastdiv_misses(b, per_binade, seed, outside, outside_bad);
}

// the create-time decision of qlnlp_create: may the kernels divide by b with the reciprocal?
int host_fastdiv_is_exact(double b) { return ql::fastdiv_is_exact(b); }
}
