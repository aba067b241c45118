"""Reference of the batched KKT solve (qlnlp_kkt_solve_batch_device), for the tests.

It assembles the full sparse KKT matrix of one problem from the handle's structure queries (qlnlp_hessian_structure,
qlnlp_jacobian_structure) and solves it with scipy.  It shares no code with the kernel: no block structure, no
elimination of the multipliers, no knot-local tables."""
import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla


def kkt_matrix(hs, hvals, js, jvals, sx, dc):
    """K = [[W + diag(sx), J'], [J, -diag(dc)]] (CSC).  hs, js: 1-based (rows, cols) of the Hessian's lower triangle
    and of the Jacobian values; the Hessian is mirrored."""
    n, m = len(sx), len(dc)
    hr, hc = np.asarray(hs[0]) - 1, np.asarray(hs[1]) - 1
    off = hr != hc
    W = sp.coo_matrix((np.concatenate([hvals, np.asarray(hvals)[off]]),
                       (np.concatenate([hr, hc[off]]), np.concatenate([hc, hr[off]]))), shape=(n, n))
    J = sp.coo_matrix((jvals, (np.asarray(js[0]) - 1, np.asarray(js[1]) - 1)), shape=(m, n))
    return sp.bmat([[W + sp.diags(sx), J.T], [J, -sp.diags(dc)]], format="csc")


def solve(K, r1, r2):
    n = len(r1)
    z = spla.spsolve(K, np.concatenate([r1, r2]))
    return z[:n], z[n:]


def residual(K, px, pl, r1, r2):
    """(||K z - r||_inf, ||K||_inf ||z||_inf + ||r||_inf) for z = [px; pl], r = [r1; r2]."""
    z, r = np.concatenate([px, pl]), np.concatenate([r1, r2])
    res = np.abs(K @ z - r).max()
    knorm = np.abs(K).sum(axis=1).max()
    return float(res), float(knorm * np.abs(z).max() + np.abs(r).max())


def schur_dense(K, n):
    """M = W + diag(sx) + J' diag(dc)^-1 J, dense, from K's blocks."""
    Kd = K.toarray()
    A, Jt, J, D = Kd[:n, :n], Kd[:n, n:], Kd[n:, :n], -np.diag(Kd[n:, n:])
    return A + Jt @ (J / D[:, None])


def status_of(M, N, tol=0.0):
    """The status the factorisation reports for a dense M: 0 if positive definite, else the first knot whose leading
    principal submatrix (knots 1..k) is not positive definite."""
    for k in range(1, N + 1):
        w = np.linalg.eigvalsh(M[:20 * k - (5 if k == N else 0), :20 * k - (5 if k == N else 0)])
        if w.min() <= tol:
            return k
    return 0
