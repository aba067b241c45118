"""Extended-precision reference of the KKT step, for the accuracy tests of the batched KKT solve.

K is the full sparse KKT matrix of tests/kkt_ref.py (kkt_matrix, the independent assembly).  kkt_solve_hp factors it
with scipy's splu, which pivots, and refines the solution with residuals computed in long double: no block structure,
no elimination of the multipliers, nothing shared with the kernel.  The x86-64 long double (64-bit significand, eps =
1.1e-19) is required; where numpy's long double is plain fp64 the caller skips."""
import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

LD = np.longdouble
EPS = float(np.finfo(np.float64).eps) / 2          # unit roundoff of fp64
STOP = 1e-18                                       # correction / solution, per block, at which refinement stops
FLOOR = 1e-16                                      # ... or below which corrections that stopped shrinking are accepted
MAX_STEPS = 10


def require_long_double():
    if not np.finfo(LD).eps < 1e-18:
        pytest.skip("numpy's long double is not an extended type here")


class NotConverged(RuntimeError):
    pass


def _csr(K):
    return sp.csr_matrix(K)


def matvec_hp(K, z):
    """K z in long double: a CSR mat-vec over K.data cast to long double, each row a left-to-right np.add.reduceat."""
    A = _csr(K)
    prod = A.data.astype(LD) * np.asarray(z, dtype=LD)[A.indices]
    out = np.zeros(A.shape[0], dtype=LD)
    nz = np.diff(A.indptr) > 0
    if prod.size:
        out[nz] = np.add.reduceat(prod, A.indptr[:-1][nz])
    return out


def residual_hp(K, z, r):
    """r - K z in long double."""
    return np.asarray(r, dtype=LD) - matvec_hp(K, z)


def abs_scale_hp(K, z, r):
    """|K| |z| + |r| in long double (the denominator of the componentwise backward error)."""
    A = _csr(K)
    return matvec_hp(sp.csr_matrix((np.abs(A.data), A.indices, A.indptr), shape=A.shape), np.abs(np.asarray(z, dtype=LD))) \
        + np.abs(np.asarray(r, dtype=LD))


def normwise_bwd(K, z, r):
    """||r - K z||_inf / (||K||_inf ||z||_inf + ||r||_inf), the residual in long double."""
    res = float(np.abs(residual_hp(K, z, r)).max())
    knorm = float(np.abs(_csr(K)).sum(axis=1).max())
    return res / (knorm * float(np.abs(np.asarray(z, dtype=LD)).max()) + float(np.abs(r).max()))


def componentwise_bwd(K, z, r):
    """Oettli-Prager: max_i |r - K z|_i / (|K| |z| + |r|)_i."""
    res = np.abs(residual_hp(K, z, r))
    den = abs_scale_hp(K, z, r)
    return float(np.max(np.where(den > 0, res / np.where(den > 0, den, 1), np.where(res > 0, np.inf, 0))))


def kkt_solve_hp(K, r, n):
    """z with K z = r to long-double accuracy: splu of K, then refinement z += LU \\ (r - K z) with the residual and z in
    long double, until the correction of each block (px = z[:n], pl = z[n:]) is below STOP of that block, in at most
    MAX_STEPS steps.  When pl is many orders larger than px, the long-double residual's own rounding (1e-19 |K| |z|)
    leaves px corrections of 1e-18 .. 1e-17 of px that no longer shrink: corrections that stall below FLOOR are accepted,
    and z is then known to about its last correction, four orders below the tightest bound the tests assert.  Raises
    NotConverged (or scipy's RuntimeError for an exactly singular K) otherwise."""
    require_long_double()
    lu = spla.splu(sp.csc_matrix(K))
    z = lu.solve(np.asarray(r, dtype=np.float64)).astype(LD)
    hist = []
    for _ in range(MAX_STEPS):
        d = lu.solve(residual_hp(K, z, r).astype(np.float64)).astype(LD)
        if not np.isfinite(d).all():
            break
        z = z + d
        rel = [float(np.abs(d[blk]).max() / np.abs(z[blk]).max()) for blk in (slice(0, n), slice(n, None))]
        hist.append("%.1e/%.1e" % tuple(rel))
        if max(rel) <= STOP:
            return z
        if len(hist) > 1 and max(rel) <= FLOOR and max(rel) >= 0.5 * prev:
            return z
        prev = max(rel)
    raise NotConverged("iterative refinement of the reference did not converge; px / pl corrections: " + " ".join(hist))


def block_errors(z, z_ref, n):
    """(px error, pl error): max |z - z_ref| / max |z_ref| over each block."""
    z, z_ref = np.asarray(z, dtype=LD), np.asarray(z_ref, dtype=LD)
    out = []
    for blk in (slice(0, n), slice(n, None)):
        out.append(float(np.abs(z[blk] - z_ref[blk]).max() / np.abs(z_ref[blk]).max()))
    return tuple(out)
