"""Lagrangian Hessian (SURVEY.md 8f N3) -- CPU side.  There is no reference target (src/moi.jl:26-28 offers
[:Grad, :Jac] only), so the chain of evidence is: the oracle's dense second-order forward mode (oracle/ql_oracle_hess.c)
is checked against a 50-digit finite-difference second derivative of the oracle's own f and g; the closed-form
structure and the generated device code (emulated on the host with the kernel's headers) are checked against that
oracle."""
import numpy as np
import pytest

from oracle import oracle as om
from oracle.oracle import Oracle
from quadruped_landing_b200 import HybridNLP, PlanarQuadruped, build_problem, initial_guess

CLASSES = [(61, 21, 1), (61, 21, 2), (31, 11, 2), (5, 3, 1), (2, 1, 1), (2, 2, 2), (33, 33, 1), (33, 1, 2), (65, 2, 1)]


def _point(prob, seed):
    rng = np.random.default_rng(seed)
    base = initial_guess(prob) if prob.k_trans > 1 else np.zeros(prob.n_nlp)
    Z = base + 5e-2 * rng.standard_normal(prob.n_nlp)
    Z[19::20] = np.clip(Z[19::20], 1e-3, 2e-2)
    lam = rng.standard_normal(prob.m_nlp)
    return Z, lam, float(rng.uniform(0.3, 1.7))


def test_rk4_hessian_against_extended_precision():
    """sum_r lam_r Hess(rk4_r): the oracle's second-order forward mode vs central second differences of the RK4 map
    evaluated in 50-digit arithmetic (the mpmath restatement in tests/mp_nlp.py), all three modes."""
    mp = pytest.importorskip("mpmath")
    from mp_nlp import rk4
    mp.mp.dps = 50
    model = PlanarQuadruped()
    rng = np.random.default_rng(5)

    for mode in (1, 2, 3):
        x = rng.standard_normal(15)
        u = np.concatenate([rng.standard_normal(4) * 30, [0.013]])
        lam = rng.standard_normal(15)
        H = om.rk4_hessian(model, mode, x, u, lam)
        assert np.array_equal(H, H.T)
        z0 = [mp.mpf(float(v)) for v in np.concatenate([x, u])]
        lm = [mp.mpf(float(v)) for v in lam]
        phi = lambda z: sum(l * o for l, o in zip(lm, rk4(mode, model, z[:15], z[15:])))
        e = mp.mpf(10) ** -12
        scale = max(1.0, np.abs(H).max())
        for (i, j) in [(19, 19), (19, 16), (19, 2), (16, 1), (15, 4), (19, 9), (17, 5), (18, 6), (19, 12), (0, 0), (3, 19), (9, 9)]:
            zi = lambda si, sj: [v + si * e * (k == i) + sj * e * (k == j) for k, v in enumerate(z0)]
            d2 = (phi(zi(1, 1)) - phi(zi(1, -1)) - phi(zi(-1, 1)) + phi(zi(-1, -1))) / (4 * e * e)
            assert abs(float(d2) - H[i, j]) <= 1e-11 * scale, (mode, i, j, float(d2), H[i, j])


@pytest.mark.parametrize("N,kt,im", CLASSES)
def test_structure_and_generated_code_against_the_oracle(emul_lib, N, kt, im):
    prob = build_problem(N=N, k_trans=kt, init_mode=im)
    nlp = HybridNLP.from_problem(prob, hessian=True)
    assert nlp.features_available() == ["Grad", "Jac", "Hess"]
    o = Oracle(prob)
    rows, cols = nlp.hessian_structure_arrays()
    assert len(rows) == nlp.nnz_hess and np.all(rows >= cols)
    lin = (cols - 1) * prob.n_nlp + rows
    assert np.all(np.diff(lin) > 0)                                  # column-major, no duplicates
    assert np.all((rows - 1) // 20 == (cols - 1) // 20)              # block diagonal: one block per knot
    m = prob.model
    worst = 0.0
    for seed in range(3):
        Z, lam, sigma = _point(prob, 100 * N + seed)
        H = o.hess_lagrangian_dense(Z, sigma, lam)
        assert np.array_equal(H, H.T)
        # everything outside the pattern is exactly zero (lower triangle)
        mask = np.zeros_like(H, dtype=bool)
        mask[rows - 1, cols - 1] = True
        assert not np.tril(H)[~mask].any()
        out = np.empty(nlp.nnz_hess)
        rc = emul_lib.emul_hess_stream(N, kt, im, m.g, m.mb, m.mf, m.lb, prob.Q.ctypes.data, prob.R.ctypes.data,
                                       prob.q.ctypes.data, prob.r.ctypes.data, Z.ctypes.data, sigma, lam.ctypes.data,
                                       out.ctypes.data, nlp.nnz_hess)
        assert rc == 0
        want = H[rows - 1, cols - 1]
        tol = 1e-12 * max(1.0, np.abs(want).max())
        assert np.abs(out - want).max() <= tol
        worst = max(worst, np.abs(out - want).max() / max(1.0, np.abs(want).max()))
    assert worst <= 1e-12


def test_default_instance_counts():
    nlp = HybridNLP.from_problem(build_problem())
    assert nlp.features_available() == ["Grad", "Jac"]                 # the reference's answer unless asked otherwise
    assert nlp.nnz_hess == 20 * 57 + 40 * 55 + 15 == 3355


def test_hessian_is_the_derivative_of_the_lagrangian_gradient():
    """Independent of second-order forward mode: central differences of grad L = sigma grad f_true + J' lambda, with J from
    the oracle and grad f_true = the TRUE gradient of eval_f (the reference's grad_f! omits d/dh, quirk Q1)."""
    prob = build_problem(N=7, k_trans=3)
    o = Oracle(prob)
    Z, lam, sigma = _point(prob, 3)

    def lagrangian(z):
        return sigma * o.eval_f(z) + lam @ o.eval_c(z)

    H = o.hess_lagrangian_dense(Z, sigma, lam)
    e = 1e-4
    rng = np.random.default_rng(0)
    for _ in range(40):
        k = rng.integers(0, 6)
        i, j = 20 * k + rng.integers(0, 20), 20 * k + rng.integers(0, 20)
        ei, ej = np.zeros_like(Z), np.zeros_like(Z)
        ei[i], ej[j] = e, e
        d2 = (lagrangian(Z + ei + ej) - lagrangian(Z + ei - ej) - lagrangian(Z - ei + ej) + lagrangian(Z - ei - ej)) / (4 * e * e)
        assert abs(d2 - H[i, j]) <= 2e-5 * max(1.0, abs(H[i, j])), (i, j, d2, H[i, j])
