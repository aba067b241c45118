"""The extended-precision KKT reference (tests/kkt_hp.py) checked on the CPU: its refined solve against a 40-digit LU of
the dense K at benign and at interior-point scalings, its long-double residual on inputs where the residual is exact, and
its refusal to return a solution of a singular K."""
import numpy as np
import pytest
import scipy.sparse as sp

from oracle.oracle import Oracle
from quadruped_landing_b200 import HybridNLP, build_problem

import kkt_hp
import kkt_ref
from test_mp_reference_cpu import perturbed
from test_second_order_cpu import spd_w

mpmath = pytest.importorskip("mpmath")


def _mp_solve(K, r):
    """K^-1 r with a 40-digit LU (mpmath, partial pivoting) of the dense K, rounded to long double."""
    with mpmath.workdps(40):
        A = mpmath.matrix(K.toarray().tolist())
        z = mpmath.lu_solve(A, mpmath.matrix([float(v) for v in r]))
        return np.array([np.longdouble(mpmath.nstr(z[i], 30)) for i in range(len(r))], dtype=np.longdouble)


def _inputs(N, kt, regime, seed):
    p = build_problem(N=N, k_trans=kt, init_mode=1)
    nlp = HybridNLP.from_problem(p, pattern="true", hessian=True)
    jv = Oracle(p).jac_c_sparse_true(perturbed(p, N + kt))
    rng = np.random.default_rng(seed)
    n, m = nlp.n_nlp, nlp.m_nlp
    lb, ub = nlp.constraint_bounds()
    if regime == "benign":
        sx, dc = rng.uniform(1.0, 10.0, n), rng.uniform(1e-2, 1.0, m)
    else:                                    # equality rows at 1e-12, the barrier diagonal over 16 decades
        sx = 10.0 ** rng.uniform(-8.0, 8.0, n)
        dc = np.where(lb == ub, 1e-12, rng.uniform(1e-2, 1.0, m))
    K = kkt_ref.kkt_matrix(nlp.hessian_structure_arrays(), spd_w(nlp, seed), nlp.jacobian_structure_arrays(), jv, sx, dc)
    return K, np.concatenate([rng.standard_normal(n), rng.standard_normal(m)]), n


@pytest.mark.parametrize("N,kt", [(2, 1), (2, 2), (3, 2)])
@pytest.mark.parametrize("regime", ["benign", "interior-point"])
def test_refined_solve_matches_a_40_digit_lu(N, kt, regime):
    kkt_hp.require_long_double()
    K, r, n = _inputs(N, kt, regime, seed=10 * N + kt)
    z = kkt_hp.kkt_solve_hp(K, r, n)
    want = _mp_solve(K, r)
    ex, el = kkt_hp.block_errors(z, want, n)
    print(f"N={N} kt={kt} {regime}: px {ex:.1e}, pl {el:.1e}")
    assert ex <= 1e-17 and el <= 1e-17, (ex, el)
    # the plain fp64 solve is not this accurate at the interior-point scaling: the reference adds digits
    z64 = np.concatenate(kkt_ref.solve(K, r[:n], r[n:]))
    assert max(kkt_hp.block_errors(z64, want, n)) > 1e-17
    assert kkt_hp.componentwise_bwd(K, z, r) <= 1e-17


def test_residual_is_exact_on_small_integers():
    kkt_hp.require_long_double()
    rng = np.random.default_rng(3)
    A = rng.integers(-9, 10, (40, 40)) * (rng.random((40, 40)) < 0.3)
    z = rng.integers(-99, 100, 40)
    r = rng.integers(-999, 1000, 40)
    K = sp.csc_matrix(A.astype(np.float64))
    want = r - A @ z                                        # Python / numpy integers: exact
    got = kkt_hp.residual_hp(K, z.astype(np.float64), r.astype(np.float64))
    assert np.array_equal(got, want.astype(np.longdouble))
    # an empty row gives r itself
    A[5] = 0
    got = kkt_hp.residual_hp(sp.csc_matrix(A.astype(np.float64)), z.astype(np.float64), r.astype(np.float64))
    assert got[5] == r[5]


def test_singular_matrix_raises():
    """Two equal rows and a right-hand side that differs on them: no z solves K z = r, and none is returned."""
    kkt_hp.require_long_double()
    K, r, n = _inputs(2, 2, "benign", seed=1)
    Kd = K.toarray()
    Kd[n + 3] = Kd[n + 7]
    r = r.copy()
    r[n + 3] = r[n + 7] + 1.0
    with pytest.raises(RuntimeError):
        kkt_hp.kkt_solve_hp(sp.csc_matrix(Kd), r, n)
    # nearly singular in fp64 (a row equal to another up to rounding): splu factors it, the refinement refuses
    Kd[n + 3] = Kd[n + 7] * (1.0 + 2.0 ** -52)
    with pytest.raises(kkt_hp.NotConverged):
        kkt_hp.kkt_solve_hp(sp.csc_matrix(Kd), r, n)


def test_stalled_refinement_is_accepted_below_the_floor_only(monkeypatch):
    """With the 1e-18 stop out of reach, the refinement ends on the stall rule (corrections below FLOOR that stopped
    shrinking) and the solution still matches a 40-digit LU; with the floor out of reach too, it raises."""
    kkt_hp.require_long_double()
    K, r, n = _inputs(2, 2, "interior-point", seed=22)
    monkeypatch.setattr(kkt_hp, "STOP", -1.0)
    z = kkt_hp.kkt_solve_hp(K, r, n)
    ex, el = kkt_hp.block_errors(z, _mp_solve(K, r), n)
    assert ex <= 1e-17 and el <= 1e-17, (ex, el)
    monkeypatch.setattr(kkt_hp, "FLOOR", -1.0)
    with pytest.raises(kkt_hp.NotConverged):
        kkt_hp.kkt_solve_hp(K, r, n)
