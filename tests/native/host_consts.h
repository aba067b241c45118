// Host-side definitions the generated header (csrc/rk4_dual_gen.h) expects from its includer.
// Plain IEEE operations; compile with -ffp-contract=off.  With -DQL_HOST_FASTDIV the divisions by the model constants
// are the kernels' reciprocal division (csrc/fastdiv.h) instead, and host_fastdiv_edges() counts the divisions whose
// numerator is outside its domain (|a| < 2^-969, or a*r overflowing), +0 aside.  TEST HARNESS ONLY.
#pragma once
#define QL_ADD(a, b) ((a) + (b))
#define QL_SUB(a, b) ((a) - (b))
#define QL_MUL(a, b) ((a) * (b))
#ifdef QL_HOST_FASTDIV
#include <cmath>
#include "../../quadruped_landing_b200/csrc/fastdiv.h"
static long long host_fastdiv_edge_count = 0;
static inline double host_fastdiv(double a, double b)
{
    const double r = 1.0 / b;
    if (!ql::fastdiv_in_domain(a, r) && (a != 0.0 || std::signbit(a))) ++host_fastdiv_edge_count;   // +0 is exact
    return ql::fastdiv(a, b, r);
}
extern "C" long long host_fastdiv_edges() { return host_fastdiv_edge_count; }
#define QL_DIV_MB(a) host_fastdiv((a), K.mb)
#define QL_DIV_MF(a) host_fastdiv((a), K.mf)
#define QL_DIV_IB(a) host_fastdiv((a), K.Ib)
#define QL_DIV_SIX(a) host_fastdiv((a), 6.0)
#else
#define QL_DIV_MB(a) ((a) / K.mb)
#define QL_DIV_MF(a) ((a) / K.mf)
#define QL_DIV_IB(a) ((a) / K.Ib)
#define QL_DIV_SIX(a) ((a) / 6.0)
#endif
#define QL_FN static inline
#define QL_ST(ptr, off, val) ((ptr)[(off)] = (val))
#define QL_PADD(ptr, n) ((ptr) + (n))
struct HostConsts {
    double g, mb, mf, Ib;
};
