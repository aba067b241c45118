"""Independent extended-precision check of the oracle's RK4 step and of its forward-mode Jacobian.

The reference records no gradient/Jacobian values ("parity unpinned", DESIGN.md section 2), so the oracle's
`qlo_rk4_jacobian` (dense ForwardDiff-style duals in fp64) is checked here against the MATHEMATICAL
derivative of the reference's RK4 map (planar_quadruped.jl:36-221), obtained from the mpmath restatement in
tests/mp_nlp.py by central differences at 60 digits (truncation error ~1e-36)."""
import numpy as np
import pytest

from oracle import oracle
from quadruped_landing_b200 import PlanarQuadruped

mp = pytest.importorskip("mpmath")
mp.mp.dps = 60
from mp_nlp import rk4  # noqa: E402


def rk4_mp(mode, m, z):
    """contactM_dynamics_rk4, planar_quadruped.jl:189-221, z = [x(15); u(5)] (the restatement in tests/mp_nlp.py)."""
    return rk4(mode, m, z[:15], z[15:])


@pytest.mark.parametrize("mode", [1, 2, 3])
def test_rk4_and_jacobian_against_extended_precision(mode):
    m = PlanarQuadruped()
    rng = np.random.default_rng(40 + mode)
    for _ in range(6):
        x = rng.normal(size=15) * np.array([0.5] * 7 + [3.0] * 7 + [0.5])
        u = np.array([*rng.normal(size=4) * 40 + np.array([0, 50, 0, 50]), rng.uniform(1e-3, 2e-2)])
        xn, J = oracle.rk4_jacobian(m, mode, x, u)
        z = [mp.mpf(float(v)) for v in np.concatenate([x, u])]
        ref = rk4_mp(mode, m, z)
        scale = 1.0 + np.abs(xn)
        assert np.all(np.abs(xn - np.array([float(r) for r in ref])) <= 8e-16 * scale)
        eps = mp.mpf(10) ** -18
        Jref = np.empty((15, 20))
        for j in range(20):
            zp, zm = list(z), list(z)
            zp[j] += eps
            zm[j] -= eps
            col = [(a - b) / (2 * eps) for a, b in zip(rk4_mp(mode, m, zp), rk4_mp(mode, m, zm))]
            Jref[:, j] = [float(c) for c in col]
        # fp64 forward mode: a few ulp of the largest term entering each entry
        tol = 1e-14 + 1e-13 * np.abs(Jref) + 2e-16 * np.abs(Jref).max()
        assert np.all(np.abs(J - Jref) <= tol), np.abs(J - Jref).max()
        # structural zeros of the analytic derivative are exact zeros in the oracle
        assert not J[np.abs(Jref) < 1e-30].any()


def test_quirks_are_deliberate(golden):
    """Q1/Q2/Q4 of SURVEY.md 8a: places where the reference is NOT the analytic derivative."""
    import quadruped_landing_b200 as ql
    p = ql.default_problem()
    o = oracle.Oracle(p)
    z = golden["data_6"].copy()
    # Q1: d f / d h_k is h_k*(R55*h_k + r5) = 0 in the default instance, although f depends on h_k
    grad = o.grad_f(z)
    assert not grad[19::20].any()
    zp = z.copy()
    zp[19] += 1e-6
    assert abs(o.eval_f(zp) - o.eval_f(z)) > 1e-9
    # Q2: at k = k_trans-1 the time row (15th) of the RK4 block is zeroed by the jump "Jacobian"
    dense = o.jac_c_dense(z)
    k = p.k_trans - 1
    row = 29 + 15 * (k - 1) + 14
    assert not dense[row, 20 * (k - 1):20 * k].any()
    assert dense[row - 15, 20 * (k - 2) + 14] == 1.0 and dense[row - 15, 20 * (k - 2) + 19] == 1.0
    # Q4: body-clearance derivative is +lb/2*cos(theta) when theta <= 0 (here theta = 0 exactly)
    z0 = ql.initial_guess(p)
    assert z0[20 * 30 + 2] == 0.0
    d0 = o.jac_c_dense(z0)
    assert d0[o.m_nlp - p.N + 30, 20 * 30 + 2] == 0.25
