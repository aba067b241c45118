"""KKT inputs built on the host with a known answer, for the GPU tests of the second-order kernels
(tests/test_gpu_second_order.py): a diagonally dominant W (M > 0 even without sx), and the same W with one negative
diagonal entry planted at knot k0, sized from a bound on diag(J' D^-1 J) so that the first leading block of M that is
not positive definite is knot k0's, whatever J and dc >= dc_min hold.  Here the construction is checked against the
dense eigenvalues of the reference (tests/kkt_ref.py), so the GPU test's expected statuses do not rest on the kernel."""
import numpy as np
import pytest

from oracle.oracle import Oracle
from quadruped_landing_b200 import HybridNLP, build_problem

import kkt_ref
from test_mp_reference_cpu import perturbed


def spd_w(nlp, seed):
    """W values in hessian_structure order: off-diagonal entries in [-1, 1], each diagonal entry 1 + the sum of the
    magnitudes of the off-diagonal entries of its row (the lower triangle mirrored)."""
    hr, hc = nlp.hessian_structure_arrays()
    w = np.random.default_rng(seed).uniform(-1.0, 1.0, len(hr))
    off = hr != hc
    rowsum = np.zeros(nlp.n_nlp)
    np.add.at(rowsum, hr[off] - 1, np.abs(w[off]))
    np.add.at(rowsum, hc[off] - 1, np.abs(w[off]))
    w[~off] = 1.0 + rowsum[hr[~off] - 1]
    return w


def w_dense(nlp, w):
    hr, hc = nlp.hessian_structure_arrays()
    W = np.zeros((nlp.n_nlp, nlp.n_nlp))
    W[hr - 1, hc - 1] = w
    W[hc - 1, hr - 1] = w
    return W


def planted_entry(nlp, k0):
    """(variable, index into the W values) of the diagonal entry planted at knot k0: a control column (local 17) before
    the last knot, a state column (local 14) at knot N, which has 15 variables."""
    i = 20 * (k0 - 1) + (17 if k0 < nlp.N else 14)
    hr, hc = nlp.hessian_structure_arrays()
    e = np.nonzero((hr == i + 1) & (hc == i + 1))[0]
    assert e.size == 1
    return i, int(e[0])


def planted_value(nlp, jv, k0, dc_min):
    """A W diagonal value that makes M's diagonal entry at the planted variable i negative for every dc >= dc_min:
    (J' D^-1 J)_ii = sum_r J_ri^2 / dc_r <= sum_r J_ri^2 / dc_min =: u, and W_ii = -(2u + 1) leaves M_ii <= -u - 1."""
    i, _ = planted_entry(nlp, k0)
    _, cols = nlp.jacobian_structure_arrays()
    u = float(np.sum(np.asarray(jv)[cols == i + 1] ** 2)) / dc_min
    return -(2.0 * u + 1.0)


def planted_w(nlp, w, jv, k0, dc_min):
    w = w.copy()
    w[planted_entry(nlp, k0)[1]] = planted_value(nlp, jv, k0, dc_min)
    return w


@pytest.mark.parametrize("N,kt,im", [(2, 2, 1), (2, 1, 2), (5, 3, 1), (9, 4, 2)])
def test_planted_status_is_the_reference_status(N, kt, im):
    p = build_problem(N=N, k_trans=kt, init_mode=im)
    nlp = HybridNLP.from_problem(p, pattern="true", hessian=True)
    hs, js = nlp.hessian_structure_arrays(), nlp.jacobian_structure_arrays()
    n = nlp.n_nlp
    jv = Oracle(p).jac_c_sparse_true(perturbed(p, N))
    rng = np.random.default_rng(N + kt)
    dc_min = 1e-2
    w = spd_w(nlp, N)
    assert np.linalg.eigvalsh(w_dense(nlp, w)).min() > 0                # W alone is positive definite
    for trial in range(3):
        dc = rng.uniform(dc_min, 1.0, nlp.m_nlp)
        if trial == 1:
            dc[:] = dc_min                   # the bound is tight on dc: the smallest dc allowed
        M = kkt_ref.schur_dense(kkt_ref.kkt_matrix(hs, w, js, jv, np.zeros(n), dc), n)
        assert kkt_ref.status_of(M, N) == 0
        for k0 in range(1, N + 1):
            M = kkt_ref.schur_dense(kkt_ref.kkt_matrix(hs, planted_w(nlp, w, jv, k0, dc_min), js, jv, np.zeros(n), dc), n)
            assert kkt_ref.status_of(M, N) == k0, (trial, k0)
            i, _ = planted_entry(nlp, k0)
            assert M[i, i] < -1.0
