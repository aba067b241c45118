"""The kernels' division by a model constant (csrc/fastdiv.h) at the ends of the double range, on the CPU.

The host twins of the generated code (tests/native/rk4_gen_host.cpp and emul_products.cpp, which between them run the
RK4 step, its Jacobian, the Jacobian products and the Lagrangian Hessian routines of csrc/rk4_dual_gen.h) are built a
second time with the kernels' reciprocal division in place of '/', and count the divisions whose numerator is outside
the formula's domain (|a| >= 2^-969, a*r finite; +0 aside, whose quotient is exact).  At inputs scaled towards the subnormals and towards
overflow:
* the IEEE build equals the oracle wherever the oracle is finite (its dense duals overflow at huge inputs where the
  sparse code does not, never the other way round);
* an input whose divisions all stay inside the domain gives the fast build the bits of the IEEE build;
* one that leaves it gives what fastdiv.h documents, carried through the step: outputs within the parity tolerance
  (1e-14 + 1e-12 |x|, +0.0 == -0.0) of the IEEE build below 2^-969, NaN where a*r overflows;
* each test requires a floor of divisions outside the domain, so that it cannot quietly stop reaching the edge."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle
from quadruped_landing_b200 import PlanarQuadruped, build_problem

from conftest import _compile_native
from test_products_cpu import _point, _vectors
from test_rk4_gen import _samples

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODELS = {"default": PlanarQuadruped(), "random": PlanarQuadruped(g=-3.71, mb=7.3, mf=0.23, lb=0.61)}
TINY = [2.0 ** -990, 2.0 ** -1000, 2.0 ** -1010, 2.0 ** -1018]
DP = C.c_void_p


def _fast_build(tmp_dir, name):
    out = os.path.join(tmp_dir, name + "_fastdiv.so")
    subprocess.run(["g++", "-O2", "-ffp-contract=off", "-DQL_HOST_FASTDIV", "-fPIC", "-shared", "-o", out,
                    os.path.join(ROOT, "tests", "native", name + ".cpp")], check=True)
    L = C.CDLL(out)
    L.host_fastdiv_edges.restype = C.c_longlong
    return L


def _rk4_argtypes(L):
    L.host_rk4_jac.argtypes = [C.c_int, DP, DP] + [C.c_double] * 4 + [DP, DP]
    L.host_rk4.argtypes = [C.c_int, DP, DP] + [C.c_double] * 4 + [DP]
    return L


def _prod_argtypes(L):
    model = [C.c_int] * 3 + [C.c_double] * 4
    L.emul_jvp.argtypes = model + [DP] * 3
    L.emul_vjp.argtypes = model + [DP] * 3
    L.emul_hvp.argtypes = model + [DP] * 5 + [C.c_double, DP, DP, DP]
    return L


@pytest.fixture(scope="module")
def fast(tmp_path_factory):
    d = str(tmp_path_factory.mktemp("fastdiv"))
    return {"rk4": _rk4_argtypes(_fast_build(d, "rk4_gen_host")), "prod": _prod_argtypes(_fast_build(d, "emul_products"))}


@pytest.fixture(scope="module")
def ieee_prod():
    return _prod_argtypes(C.CDLL(_compile_native("emul_products")))


def assert_bits(got, want, what):
    """The same bits, NaN for NaN (payloads aside)."""
    got, want = np.asarray(got), np.asarray(want)
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan), (what, np.argwhere(np.isnan(got) != nan)[:4].tolist())
    bad = got.view(np.int64) != want.view(np.int64)
    bad &= ~nan
    assert not bad.any(), (what, np.argwhere(bad)[:4].tolist(), got[bad][:4], want[bad][:4])


def assert_equal_where_finite(got, want, what):
    """The oracle's parity rule (tests/test_rk4_gen.py): equal values, +0.0 == -0.0, wherever the oracle is finite."""
    fin = np.isfinite(want)
    assert np.array_equal(got[fin], want[fin]), (what, np.argwhere(fin & (got != want))[:4].tolist())


def assert_documented(fast, ieee, left_domain, huge, what):
    """The fast build against the IEEE build: the same bits while every division stayed inside the domain; else NaN
    (a*r overflowing: huge inputs) or the parity tolerance (numerators below 2^-969) where the two differ."""
    if not left_domain:
        assert_bits(fast, ieee, what)
        return
    differ = fast.view(np.int64) != ieee.view(np.int64)
    differ &= ~(np.isnan(fast) & np.isnan(ieee))
    assert np.isnan(fast[np.isnan(ieee)]).all(), what
    if huge:
        assert np.isnan(fast[differ]).all(), (what, fast[differ][:4], ieee[differ][:4])
    else:
        a, b = fast[differ], ieee[differ]
        assert np.all(np.abs(a - b) <= 1e-14 + 1e-12 * np.abs(b)), (what, a[:4], b[:4])


def huge_forces(rng, n):
    """Forces of magnitude 1e306 to 1.5e308, random signs: a*r overflows in some divisions (by mf and Ib), where the
    unguarded correction forms Inf - Inf."""
    return np.minimum(10.0 ** rng.uniform(306, 308.2, n), 1.5e308) * np.where(rng.random(n) < 0.5, -1.0, 1.0)


def edge_inputs(seed):
    """(kind, x, u): x, u and h scaled towards the subnormals; single entries at subnormals and -0.0; huge forces."""
    rng = np.random.default_rng(seed)
    for t, (x, u) in enumerate(_samples(60, seed)):
        for s in TINY:
            yield "tiny", x * s, u * s
        xs, us = x.copy(), u.copy()
        i = rng.integers(0, 20)
        v = [5e-324, -5e-324, 2.0 ** -1060, -2.0 ** -1030, 2.0 ** -1022, -0.0][t % 6]
        if i < 15:
            xs[i] = v
        else:
            us[i - 15] = v
        yield "entry", xs, us
        uf = u.copy()
        uf[:4] = huge_forces(rng, 4)
        yield "huge", x, uf


@pytest.mark.parametrize("model", sorted(MODELS))
@pytest.mark.parametrize("mode", [1, 2, 3])
def test_rk4_and_jacobian_at_the_ends_of_the_range(fast, rk4_host_lib, model, mode):
    m = MODELS[model]
    L = fast["rk4"]
    args = (m.g, m.mb, m.mf, m.lb)
    edges = {"tiny": 0, "entry": 0, "huge": 0}
    for kind, x, u in edge_inputs(10 * mode + len(model)):
        before = L.host_fastdiv_edges()
        out = {}
        for name, lib in (("fast", L), ("ieee", rk4_host_lib)):
            xn, J, xv = np.empty(15), np.empty(300), np.empty(15)
            lib.host_rk4_jac(mode, x.ctypes.data, u.ctypes.data, *args, xn.ctypes.data, J.ctypes.data)
            lib.host_rk4(mode, x.ctypes.data, u.ctypes.data, *args, xv.ctypes.data)
            out[name] = (xn, J.reshape(20, 15).T, xv)
        left = L.host_fastdiv_edges() - before
        edges[kind] += left
        for got, want, what in zip(out["fast"], out["ieee"], ("xn", "J", "rk4")):
            assert_documented(got, want, left > 0, kind == "huge", (kind, what))
        xn0, J0 = oracle.rk4_jacobian(m, mode, x, u)
        xn, J, xv = out["ieee"]
        assert_equal_where_finite(xn, xn0, (kind, "xn vs oracle"))
        assert_equal_where_finite(J, J0, (kind, "J vs oracle"))
        assert_equal_where_finite(xv, oracle.rk4(m, mode, x, u), (kind, "rk4 vs oracle"))
    # the inputs still leave the domain (thousands of divisions per kind when this test was written)
    assert edges["tiny"] >= 1000 and edges["entry"] >= 10 and edges["huge"] >= 100, edges


def _scaled_points(prob, seed):
    z = _point(prob, seed)
    for s in TINY:
        yield "tiny", z * s
    zf = z.copy()
    rng = np.random.default_rng(seed)
    for k in range(prob.N - 1):
        zf[20 * k + 15:20 * k + 19] = huge_forces(rng, 4)
    yield "huge", zf
    ze = z.copy()
    ze[rng.integers(0, prob.n_nlp, 12)] = [5e-324, -5e-324, 2.0 ** -1060, -0.0] * 3
    yield "entry", ze


@pytest.mark.parametrize("N,kt,im", [(2, 1, 1), (33, 1, 2), (61, 21, 1), (61, 21, 2)])
def test_products_and_hessian_at_the_ends_of_the_range(fast, ieee_prod, N, kt, im):
    """J w, J' y and H v: the generated jvp / vjp / Hessian routines of the fast build against the IEEE build."""
    prob = build_problem(N=N, k_trans=kt, init_mode=im)
    m = prob.model
    args = (N, kt, im, m.g, m.mb, m.mf, m.lb)
    w, y, v, lam, sigma = _vectors(prob, N)
    L = fast["prod"]
    edges = {"tiny": 0, "entry": 0, "huge": 0}
    for kind, Z in _scaled_points(prob, N + kt):
        before = L.host_fastdiv_edges()
        out = {}
        for name, lib in (("fast", L), ("ieee", ieee_prod)):
            jw, jty, hv = np.empty(prob.m_nlp), np.empty(prob.n_nlp), np.empty(prob.n_nlp)
            assert lib.emul_jvp(*args, Z.ctypes.data, w.ctypes.data, jw.ctypes.data) == 0
            assert lib.emul_vjp(*args, Z.ctypes.data, y.ctypes.data, jty.ctypes.data) == 0
            assert lib.emul_hvp(*args, prob.Q.ctypes.data, prob.R.ctypes.data, prob.q.ctypes.data, prob.r.ctypes.data,
                                Z.ctypes.data, sigma, lam.ctypes.data, v.ctypes.data, hv.ctypes.data) == 0
            out[name] = (jw, jty, hv)
        left = L.host_fastdiv_edges() - before
        edges[kind] += left
        for got, want, what in zip(out["fast"], out["ieee"], ("J w", "J' y", "H v")):
            assert_documented(got, want, left > 0, kind == "huge", (kind, what))
    assert edges["tiny"] >= 100 * (N - 1) and edges["huge"] >= 3 * (N - 1), edges
