"""The generated sparsity-exploiting RK4/dual code (csrc/rk4_dual_gen.h, compiled for the host by
tests/native/rk4_gen_host.cpp) must equal the oracle's dense 20-wide dual evaluation BIT FOR BIT."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle
from quadruped_landing_b200 import PlanarQuadruped

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _samples(n, seed):
    rng = np.random.default_rng(seed)
    for t in range(n):
        x = rng.normal(size=15) * np.array([1.0] * 7 + [5.0] * 7 + [1.0])
        u = rng.normal(size=5) * np.array([50.0, 50.0, 50.0, 50.0, 0.0]) + np.array([0.0, 50.0, 0.0, 50.0, 0.0])
        u[4] = rng.uniform(1e-3, 2e-2)
        if t % 3 == 0:
            x = np.round(x, 1)          # exact cancellations (x1 == xb etc.)
        if t % 7 == 0:
            u[:4] = np.round(u[:4])
        yield x, u


@pytest.mark.parametrize("mode", [1, 2, 3])
def test_generated_jacobian_bit_identical(rk4_host_lib, mode):
    m = PlanarQuadruped()
    for x, u in _samples(1500, 100 + mode):
        xn0, J0 = oracle.rk4_jacobian(m, mode, x, u)
        xn, J = np.empty(15), np.empty(300)
        rk4_host_lib.host_rk4_jac(mode, x.ctypes.data, u.ctypes.data, m.g, m.mb, m.mf, m.lb, xn.ctypes.data, J.ctypes.data)
        assert np.array_equal(xn, xn0)
        assert np.array_equal(J.reshape(20, 15).T, J0)           # +0.0 == -0.0: sign of zero is not parity
        xv = np.empty(15)
        rk4_host_lib.host_rk4(mode, x.ctypes.data, u.ctypes.data, m.g, m.mb, m.mf, m.lb, xv.ctypes.data)
        assert np.array_equal(xv, oracle.rk4(m, mode, x, u))


@pytest.mark.parametrize("mode,nnz", [(1, 71), (2, 71), (3, 57)])
def test_pattern_sizes(mode, nnz):
    """SURVEY.md 8a: true nnz of the 15x20 block is 71/71/57 for modes 1/2/3."""
    m = PlanarQuadruped()
    cnt = np.zeros((15, 20), dtype=bool)
    for x, u in _samples(50, 7):
        _, J = oracle.rk4_jacobian(m, mode, x + 0.123, u + 0.321)
        cnt |= J != 0
    assert cnt.sum() == nnz


def test_other_model_constants(rk4_host_lib):
    m = PlanarQuadruped(g=-3.71, mb=7.3, mf=0.23, lb=0.61)
    for mode in (1, 2, 3):
        for x, u in _samples(200, 5):
            xn0, J0 = oracle.rk4_jacobian(m, mode, x, u)
            xn, J = np.empty(15), np.empty(300)
            rk4_host_lib.host_rk4_jac(mode, x.ctypes.data, u.ctypes.data, m.g, m.mb, m.mf, m.lb, xn.ctypes.data, J.ctypes.data)
            assert np.array_equal(xn, xn0) and np.array_equal(J.reshape(20, 15).T, J0)


@pytest.mark.parametrize("b", [10.0, 0.1, 10.0 * (0.5 * 0.5) / 12, 6.0, 7.3, 0.23, 3.0, 1.9999999999999998])
def test_reciprocal_fma_division_is_correctly_rounded(rk4_host_lib, b):
    """The kernel divides by model constants with csrc/fastdiv.h: q' = fma(fma(-q, b, a), r, q) for q = a*r and
    r = RN(1/b).  Whenever the create-time check (fastdiv_is_exact) accepts b, q' must have the bits of the IEEE
    quotient the reference computes for 2,000 numerators of every binade inside the domain |a| >= 2^-969, a*r finite
    (signed zeros and Inf included), and do what fastdiv.h states outside it: one ulp at most below 2^-969, +0 for a
    zero numerator, NaN where a*r overflows.  The check must refuse 1.9999999999999998, whose significand is all ones."""
    import ctypes as C
    fn = rk4_host_lib.host_count_fastdiv_mismatches
    fn.restype = C.c_longlong
    fn.argtypes = [C.c_double, C.c_int, C.c_ulonglong, C.c_void_p, C.c_void_p]
    rk4_host_lib.host_fastdiv_is_exact.argtypes = [C.c_double]
    exact = bool(rk4_host_lib.host_fastdiv_is_exact(b))
    assert exact == (b != 1.9999999999999998)
    if exact:
        outside, outside_bad = C.c_longlong(0), C.c_longlong(0)
        assert fn(b, 2000, 2024, C.addressof(outside), C.addressof(outside_bad)) == 0
        assert outside.value >= 2000 * 53 and outside_bad.value == 0, (outside.value, outside_bad.value)


def test_committed_header_is_up_to_date(tmp_path):
    gen = os.path.join(ROOT, "tools", "gen_rk4_dual.py")
    hdr = os.path.join(ROOT, "quadruped_landing_b200", "csrc", "rk4_dual_gen.h")
    code = open(gen).read().replace('OUT = os.path.join(HERE, "..", "quadruped_landing_b200", "csrc", "rk4_dual_gen.h")',
                                    f'OUT = {str(tmp_path / "gen.h")!r}')
    script = tmp_path / "gen.py"
    script.write_text(code)
    subprocess.run([sys.executable, str(script)], check=True, capture_output=True)
    assert (tmp_path / "gen.h").read_text() == open(hdr).read()
