"""Extended-precision model of the landing NLP, written from SURVEY.md section 8a (blocks, layout, quirks Q1-Q4) and
the kinematic-row definition in include/qlnlp.h only.  It shares no code with oracle/ or the generated device code, so
an error that the oracle and the kernels share shows up as a difference from this model.

Values are computed in mpmath at DPS digits.  Derivatives are forward differences in that precision (step 1e-25 for
first, 1e-18 for second derivatives), which leaves an error far below fp64 rounding: every RK4 output is a polynomial
in the knot's variables.  Everything is local to a knot, so the cost is linear in the number of knots asked for:
knot k touches only the init rows (k = 1), the term rows (k = N), dynamics steps k-1 and k, its own contact, body and
kinematic rows and the final-control row (k = N-1).

Indices here are 0-based; knots are numbered 1..N as in the reference."""
import mpmath as mp
import numpy as np

DPS = 60
EPS = np.finfo(np.float64).eps
NX, NU, NZK = 15, 5, 20
JUMP_ZEROED = (4, 6, 10, 11, 12, 13)          # y1, y2 and the four foot velocities (jump map, SURVEY.md 8a A7)

_E1 = mp.mpf(10) ** -25                        # first-derivative step
_E2 = mp.mpf(10) ** -18                        # second-derivative step


def field(mode, model, x, u):
    """contact{1,2,3}_dynamics on mpmath numbers: x has 14 (or more) entries, u 5.  Mode 1 pins foot 1, mode 2 pins
    foot 2, mode 3 pins both; theta does not enter."""
    g, mb, mf, lb = (mp.mpf(float(v)) for v in (model.g, model.mb, model.mf, model.lb))
    Ib = mb * lb * lb / 12
    xb, yb, x1, y1, x2, y2 = x[0], x[1], x[3], x[4], x[5], x[6]
    F1x, F1y, F2x, F2y = u[0], u[1], u[2], u[3]
    tau = -F1x * (y1 - yb) + F1y * (x1 - xb) - F2x * (y2 - yb) + F2y * (x2 - xb)
    xd = [mp.mpf(0)] * 14
    xd[0], xd[1], xd[2] = x[7], x[8], x[9]
    xd[7], xd[8], xd[9] = (F1x + F2x) / mb, (F1y + F2y) / mb + g, tau / Ib
    if mode == 1:
        xd[5], xd[6], xd[12], xd[13] = x[12], x[13], -F2x / mf, -F2y / mf + g
    elif mode == 2:
        xd[3], xd[4], xd[10], xd[11] = x[10], x[11], -F1x / mf, -F1y / mf + g
    return xd


def rk4(mode, model, x, u, with_scale=False):
    """One classic RK4 step with step h = u[4]; the 15th output is t + h.  With ``with_scale`` also returns, per
    output, the magnitude of what the update adds: |x_i| + |h|/6 (|k1| + 2|k2| + 2|k3| + |k4|)."""
    h = u[4]
    f1 = field(mode, model, x, u)
    f2 = field(mode, model, [x[i] + h / 2 * f1[i] for i in range(14)], u)
    f3 = field(mode, model, [x[i] + h / 2 * f2[i] for i in range(14)], u)
    f4 = field(mode, model, [x[i] + h * f3[i] for i in range(14)], u)
    xn = [x[i] + h / 6 * (f1[i] + 2 * f2[i] + 2 * f3[i] + f4[i]) for i in range(14)] + [x[14] + h]
    if not with_scale:
        return xn
    sc = [abs(x[i]) + abs(h) / 6 * (abs(f1[i]) + 2 * abs(f2[i]) + 2 * abs(f3[i]) + abs(f4[i])) for i in range(14)]
    return xn, sc + [abs(x[14]) + abs(h)]


class Model:
    """The NLP of one problem (``ProblemData`` fields) at one set of boundary states.

    Rows (0-based starts): init 15 | term 14 | dyn 15(N-1) | contact-first N | contact-other N-k_trans+1 |
    final-control 1 | body N | kinematic 2N (when switched on; rows 2(k-1), 2(k-1)+1 of the block for knot k)."""

    def __init__(self, prob, x0=None, xf=None, kinematics=False):
        self.N, self.kt, self.im = int(prob.N), int(prob.k_trans), int(prob.init_mode)
        self.model = prob.model
        self.kin = bool(kinematics)
        M = lambda a: [mp.mpf(float(v)) for v in np.ravel(a)]
        self.x0 = M(prob.x0 if x0 is None else x0)
        self.xf = M(prob.xf if xf is None else xf)
        self.Q, self.R, self.q, self.r = (np.asarray(a, dtype=np.float64) for a in (prob.Q, prob.R, prob.q, prob.r))
        self.c = np.asarray(prob.c, dtype=np.float64)
        self.mbg = mp.mpf(float(prob.model.mb)) * mp.mpf(float(prob.model.g))
        self.half_lb = mp.mpf(float(prob.model.lb)) / 2
        N, kt = self.N, self.kt
        self.n = 20 * N - 5
        self.c_init, self.c_term, self.c_dyn = 0, 15, 29
        self.c_cfirst = 29 + 15 * (N - 1)
        self.c_cother = self.c_cfirst + N
        self.c_fctrl = self.c_cother + N - kt + 1
        self.c_body = self.c_fctrl + 1
        self.c_kin = self.c_body + N
        self.m = self.c_kin + (2 * N if self.kin else 0)
        self.fi, self.oi = (4, 6) if self.im == 1 else (6, 4)
        self._memo = {}

    # ---- helpers
    def mode(self, k):
        """RK4 mode of the step from knot k to k+1."""
        return 3 if k >= self.kt else self.im

    def nvar(self, k):
        return NX if k == self.N else NZK

    def _vars(self, z, k):
        return [mp.mpf(float(v)) for v in z[20 * (k - 1):20 * (k - 1) + self.nvar(k)]]

    def _step(self, k, v, with_scale=False):
        """RK4 of step k (knot k -> k+1) with the jump map applied at k = k_trans - 1."""
        out = rk4(self.mode(k), self.model, v[:NX], v[NX:], with_scale)
        xn = out[0] if with_scale else out
        if k == self.kt - 1:
            for i in JUMP_ZEROED:
                xn[i] = mp.mpf(0)
        return out

    def _cost(self, k, v):
        """h_k * stagecost_k for k < N, termcost_N at k = N, and the sum of the magnitudes of its summands."""
        Q, q = self.Q[k - 1], self.q[k - 1]
        parts = [mp.mpf(float(Q[i])) * v[i] * v[i] / 2 for i in range(NX)] + \
                [mp.mpf(float(q[i])) * v[i] for i in range(NX)] + [mp.mpf(float(self.c[k - 1]))]
        if k < self.N:
            R, r = self.R[k - 1], self.r[k - 1]
            u = v[NX:]
            parts += [mp.mpf(float(R[i])) * u[i] * u[i] / 2 for i in range(NU)] + \
                     [mp.mpf(float(r[i])) * u[i] for i in range(NU)]
            h = u[4]
            return h * mp.fsum(parts), abs(h) * mp.fsum(abs(a) for a in parts)
        return mp.fsum(parts), mp.fsum(abs(a) for a in parts)

    def rows_of_knot(self, k):
        """The rows that depend on the variables of knot k, ascending."""
        N, kt = self.N, self.kt
        rows = []
        if k == 1:
            rows += range(self.c_init, self.c_init + 15)
        if k == N:
            rows += range(self.c_term, self.c_term + 14)
        if k >= 2:
            rows += range(self.c_dyn + 15 * (k - 2), self.c_dyn + 15 * (k - 1))
        if k <= N - 1:
            rows += range(self.c_dyn + 15 * (k - 1), self.c_dyn + 15 * k)
        rows.append(self.c_cfirst + k - 1)
        if k >= kt:
            rows.append(self.c_cother + k - kt)
        if k == N - 1:
            rows.append(self.c_fctrl)
        rows.append(self.c_body + k - 1)
        if self.kin:
            rows += [self.c_kin + 2 * (k - 1), self.c_kin + 2 * (k - 1) + 1]
        return sorted(rows)

    def _local(self, k, v):
        """The rows of ``rows_of_knot(k)`` as functions of knot k's variables (terms that do not depend on them, such
        as x_{k+1} in the defect of step k, are left out: they do not change the derivative)."""
        N, kt = self.N, self.kt
        val = {}
        if k == 1:
            for i in range(15):
                val[self.c_init + i] = v[i] - self.x0[i]
        if k == N:
            for i in range(14):
                val[self.c_term + i] = v[i] - self.xf[i]
        if k >= 2:
            for i in range(15):
                val[self.c_dyn + 15 * (k - 2) + i] = -v[i]
        if k <= N - 1:
            xn = self._step(k, v)
            for i in range(15):
                val[self.c_dyn + 15 * (k - 1) + i] = xn[i]
        val[self.c_cfirst + k - 1] = v[self.fi]
        if k >= kt:
            val[self.c_cother + k - kt] = v[self.oi]
        if k == N - 1:
            val[self.c_fctrl] = v[16] + v[18] + self.mbg
        val[self.c_body + k - 1] = v[1] - self.half_lb * abs(mp.sin(v[2]))
        if self.kin:
            val[self.c_kin + 2 * (k - 1)] = mp.sqrt((v[0] - v[3]) ** 2 + (v[1] - v[4]) ** 2)
            val[self.c_kin + 2 * (k - 1) + 1] = mp.sqrt((v[0] - v[5]) ** 2 + (v[1] - v[6]) ** 2)
        return [val[r] for r in self.rows_of_knot(k)]

    # ---- f and the reference gradient
    def f(self, z):
        """(f, per-knot terms, per-knot magnitude of the summands of each term)."""
        with mp.workdps(DPS):
            terms, scales = zip(*(self._cost(k, self._vars(z, k)) for k in range(1, self.N + 1)))
            return float(mp.fsum(terms)), np.array([float(t) for t in terms]), np.array([float(s) for s in scales])

    def grad(self, z):
        """(reference gradient, per-entry error scale): the derivative of f, except that d/dh_k is h(R55 h + r5) (Q1)."""
        out, sc = np.zeros(self.n), np.zeros(self.n)
        with mp.workdps(DPS):
            for k in range(1, self.N + 1):
                v = self._vars(z, k)
                h = v[19] if k < self.N else mp.mpf(1)
                o = 20 * (k - 1)
                for i in range(NX):
                    a, b = mp.mpf(float(self.Q[k - 1][i])) * v[i], mp.mpf(float(self.q[k - 1][i]))
                    out[o + i], sc[o + i] = float(h * (a + b)), float(abs(h) * (abs(a) + abs(b)))
                if k < self.N:
                    for i in range(NU):
                        a, b = mp.mpf(float(self.R[k - 1][i])) * v[NX + i], mp.mpf(float(self.r[k - 1][i]))
                        out[o + NX + i], sc[o + NX + i] = float(h * (a + b)), float(abs(h) * (abs(a) + abs(b)))
        return out, sc

    def grad_h_true(self, z, k):
        """The mathematical d f / d h_k, which the reference does not report (Q1)."""
        with mp.workdps(DPS):
            v = self._vars(z, k)
            f0 = self._cost(k, v)[0]
            v[19] += _E1
            return float((self._cost(k, v)[0] - f0) / _E1)

    # ---- g
    def g(self, z, knots=None):
        """(rows, values, scales) of the rows owned by ``knots`` (default all): knot k owns dynamics step k, its contact,
        body and kinematic rows, the init rows (k = 1), the term rows (k = N) and the final-control row (k = N-1).
        The scale of a row is the magnitude of its operands, which the row may cancel to far below (x_{k+1} and the
        RK4 update in a defect)."""
        rows, vals, scs = [], [], []
        for k in (range(1, self.N + 1) if knots is None else sorted(set(knots))):
            r, v, s = self._cached(("g", k, z[20 * (k - 1):20 * (k + 1)].tobytes()), lambda: self._g_knot(z, k))
            rows += r
            vals += v
            scs += s
        order = np.argsort(rows)
        return np.array(rows)[order], np.array(vals)[order], np.array(scs)[order]

    def _g_knot(self, z, k):
        N, kt = self.N, self.kt
        rows, vals, scs = [], [], []

        def put(r, val, s):
            rows.append(r), vals.append(float(val)), scs.append(float(s))

        with mp.workdps(DPS):
            v = self._vars(z, k)
            if k == 1:
                for i in range(15):
                    put(self.c_init + i, v[i] - self.x0[i], abs(v[i]) + abs(self.x0[i]))
            if k == N:
                for i in range(14):
                    put(self.c_term + i, v[i] - self.xf[i], abs(v[i]) + abs(self.xf[i]))
            if k < N:
                xn, sc = self._step(k, v, with_scale=True)
                nxt = self._vars(z, k + 1)
                for i in range(15):
                    put(self.c_dyn + 15 * (k - 1) + i, xn[i] - nxt[i], sc[i] + abs(nxt[i]))
            put(self.c_cfirst + k - 1, v[self.fi], abs(v[self.fi]))
            if k >= kt:
                put(self.c_cother + k - kt, v[self.oi], abs(v[self.oi]))
            if k == N - 1:
                put(self.c_fctrl, v[16] + v[18] + self.mbg, abs(v[16]) + abs(v[18]) + abs(self.mbg))
            s = self.half_lb * abs(mp.sin(v[2]))
            put(self.c_body + k - 1, v[1] - s, abs(v[1]) + s)
            if self.kin:
                for j, (a, b) in enumerate(((3, 4), (5, 6))):
                    d = mp.sqrt((v[0] - v[a]) ** 2 + (v[1] - v[b]) ** 2)
                    put(self.c_kin + 2 * (k - 1) + j, d, d)
        return rows, vals, scs

    def _cached(self, key, compute):
        """Results depend only on the variables named in ``key``: several entry points checked at the same vector
        reuse them."""
        if key not in self._memo:
            self._memo[key] = compute()
        return self._memo[key]

    # ---- reference Jacobian
    def jac_knot(self, z, k):
        """(rows, J[len(rows), nvar(k)], per-row scale) for the columns of knot k: the derivative of g with Q2 (the time
        row of the jump knot's RK4 block is 0) and Q4 (body row: d/dtheta = -lb/2 cos(theta) if theta > 0, else
        +lb/2 cos(theta)) applied.  The scale of a row is its largest entry in these columns: forward mode adds terms
        of that size."""
        return self._cached(("J", k, z[20 * (k - 1):20 * k].tobytes()), lambda: self._jac_knot(z, k))

    def _jac_knot(self, z, k):
        rows = self.rows_of_knot(k)
        with mp.workdps(DPS):
            v = self._vars(z, k)
            base = self._local(k, v)
            J = np.zeros((len(rows), self.nvar(k)))
            for j in range(self.nvar(k)):
                vp = list(v)
                vp[j] += _E1
                J[:, j] = [float((a - b) / _E1) for a, b in zip(self._local(k, vp), base)]
            br = rows.index(self.c_body + k - 1)
            th = v[2]
            J[br, 2] = float(-self.half_lb * mp.cos(th) if th > 0 else self.half_lb * mp.cos(th))
        if k == self.kt - 1:
            J[rows.index(self.c_dyn + 15 * (k - 1) + 14), :] = 0.0
        return np.array(rows), J, np.abs(J).max(axis=1)

    # ---- Lagrangian Hessian
    def hess_knot(self, z, k, sigma, lam):
        """The 20x20 (15x15 at k = N) block of sigma Hess f + sum_r lam_r Hess g_r at knot k: the true second
        derivatives (d/dh of h * stagecost included).  Linear rows contribute nothing; the body row contributes the
        theta-derivative of its Q4 Jacobian entry at (theta, theta): lam * lb/2 sin(theta) if theta > 0, else
        -lam * lb/2 sin(theta).  That is lam * lb/2 |sin(theta)| while |theta| < pi, and differs from it beyond."""
        assert not self.kin, "the Hessian covers the NLP without kinematic rows"
        lam = np.asarray(lam, dtype=np.float64)
        lk = np.concatenate([lam[self.c_dyn + 15 * (k - 1):self.c_dyn + 15 * k] if k < self.N else [], lam[self.c_body + k - 1:][:1]])
        return self._cached(("H", k, z[20 * (k - 1):20 * k].tobytes(), float(sigma), lk.tobytes()),
                            lambda: self._hess_knot(z, k, sigma, lam))

    def _hess_knot(self, z, k, sigma, lam):
        nv = self.nvar(k)
        with mp.workdps(DPS):
            v = self._vars(z, k)
            sig = mp.mpf(float(sigma))
            ld = [mp.mpf(float(lam[self.c_dyn + 15 * (k - 1) + i])) for i in range(15)] if k < self.N else []

            def phi(w):
                s = sig * self._cost(k, w)[0]
                if k < self.N:
                    s += mp.fsum(a * b for a, b in zip(ld, self._step(k, w)))
                return s

            def at(i, j):
                w = list(v)
                if i is not None:
                    w[i] += _E2
                if j is not None:
                    w[j] += _E2
                return phi(w)

            p0 = phi(v)
            p1 = [at(i, None) for i in range(nv)]
            H = np.zeros((nv, nv))
            for i in range(nv):
                for j in range(i + 1):
                    H[i, j] = H[j, i] = float((at(i, j) - p1[i] - p1[j] + p0) / (_E2 * _E2))
            th = v[2]
            H[2, 2] += float(mp.mpf(float(lam[self.c_body + k - 1])) * self.half_lb * (mp.sin(th) if th > 0 else -mp.sin(th)))
        return H


# ---- comparisons.  Every tolerance is per entry: the fp64 north star |a - b| <= 1e-14 + 1e-12 |ref|, widened only by
# a multiple of eps times the error scale the model reports for that entry (its row's operands for g, its row's largest
# entry in the knot's columns for the Jacobian, its knot block's largest entry for the Hessian).
ATOL, RTOL = 1e-14, 1e-12
G_ULPS, J_ULPS, H_ULPS = 8, 4, 16
ZERO_J = 1e-30                  # |model entry| below this: not a non-zero (first differences are exact where z_j is absent)
ZERO_H = 1e-18                  # ... relative to the block: second differences leave ~1e-24 where z_i, z_j do not meet


def sample_knots(N, k_trans, every=12):
    """All knots of a short horizon; for a long one the first knots, every 32-knot pass boundary (32j, 32j+1), the jump
    knot and its neighbours, the last two knots."""
    if N <= every:
        return list(range(1, N + 1))
    ks = {1, 2, k_trans - 1, k_trans, k_trans + 1, N - 1, N}
    for j in range(1, N // 32 + 1):
        ks |= {32 * j, 32 * j + 1}
    return sorted(k for k in ks if 1 <= k <= N)


def _fail(what, got, want, tol, idx):
    bad = np.nonzero(~(np.abs(got - want) <= tol))[0]
    if bad.size:
        i = bad[:4]
        raise AssertionError(f"{what}: {bad.size} entries off the model, first at {np.asarray(idx)[i].tolist()}: "
                             f"got {got[i].tolist()} want {want[i].tolist()} tol {np.broadcast_to(tol, got.shape)[i].tolist()}")


def check_f(m, z, f):
    """f is a sequential sum of N terms, each a sum of 41 products: the bound is (N + 48) eps times the sum of the
    magnitudes of all the summands."""
    want, _, scales = m.f(z)
    tol = (m.N + 48) * EPS * scales.sum()
    assert abs(float(f) - want) <= tol, f"f: got {float(f)!r} want {want!r} tol {tol:.3g}"


def check_grad(m, z, grad):
    want, sc = m.grad(z)
    _fail("grad", np.asarray(grad, dtype=np.float64), want, ATOL + RTOL * np.abs(want) + G_ULPS * EPS * sc, np.arange(m.n))


def check_g(m, z, g, knots=None):
    rows, want, sc = m.g(z, knots)
    _fail("g", np.asarray(g, dtype=np.float64)[rows], want, ATOL + RTOL * np.abs(want) + G_ULPS * EPS * sc, rows)


def check_jac(m, z, vals, rows, cols, knots):
    """``vals`` in the order of the 1-based (``rows``, ``cols``) pattern, which is column-major: the entries of knot k's
    columns are compared with the model, and every non-zero of the model there must be an entry of the pattern."""
    vals = np.asarray(vals, dtype=np.float64)
    for k in knots:
        lo, hi = np.searchsorted(cols, [20 * (k - 1) + 1, 20 * (k - 1) + m.nvar(k) + 1])
        r, c = rows[lo:hi] - 1, cols[lo:hi] - 1 - 20 * (k - 1)
        mr, J, sc = m.jac_knot(z, k)
        full, scale = np.zeros((m.m, m.nvar(k))), np.zeros(m.m)
        full[mr], scale[mr] = J, sc
        want = full[r, c]
        _fail(f"jac knot {k}", vals[lo:hi], want, ATOL + RTOL * np.abs(want) + J_ULPS * EPS * scale[r],
              np.stack([r + 1, c + 1 + 20 * (k - 1)], 1))
        present = np.zeros(full.shape, dtype=bool)
        present[r, c] = True
        miss = np.argwhere((np.abs(full) > ZERO_J) & ~present)
        assert miss.size == 0, f"jac knot {k}: model non-zeros outside the pattern at (row, col) {(miss[:4] + [1, 1 + 20 * (k - 1)]).tolist()}"


def check_jac_dense(m, z, dense, knots):
    """The full m x n grid (zeros included): knot k's columns against the model."""
    for k in knots:
        mr, J, sc = m.jac_knot(z, k)
        want, scale = np.zeros((m.m, m.nvar(k))), np.zeros((m.m, 1))
        want[mr], scale[mr, 0] = J, sc
        got = np.asarray(dense, dtype=np.float64)[:, 20 * (k - 1):20 * (k - 1) + m.nvar(k)]
        tol = ATOL + RTOL * np.abs(want) + J_ULPS * EPS * scale
        bad = np.argwhere(~(np.abs(got - want) <= tol))
        assert bad.size == 0, f"dense jac knot {k}: {len(bad)} entries off the model, first (row, col) " \
                              f"{(bad[:4] + [1, 1 + 20 * (k - 1)]).tolist()}"


def check_hess(m, z, sigma, lam, vals, rows, cols, knots):
    """``vals`` in the order of the 1-based lower-triangle pattern (``rows``, ``cols``); per knot block, like check_jac."""
    vals = np.asarray(vals, dtype=np.float64)
    for k in knots:
        o, nv = 20 * (k - 1), m.nvar(k)
        lo, hi = np.searchsorted(cols, [o + 1, o + nv + 1])
        r, c = rows[lo:hi] - 1 - o, cols[lo:hi] - 1 - o
        assert np.all((r >= c) & (r < nv)), f"hess knot {k}: pattern leaves the block's lower triangle"
        H = m.hess_knot(z, k, sigma, lam)
        scale = np.abs(H).max()
        want = H[r, c]
        _fail(f"hess knot {k}", vals[lo:hi], want, ATOL + RTOL * np.abs(want) + H_ULPS * EPS * scale,
              np.stack([r + 1 + o, c + 1 + o], 1))
        present = np.zeros(H.shape, dtype=bool)
        present[r, c] = True
        miss = np.argwhere(np.tril(np.abs(H) > ZERO_H * (1 + scale)) & ~present)
        assert miss.size == 0, f"hess knot {k}: model non-zeros outside the pattern at {(miss[:4] + 1 + o).tolist()}"
