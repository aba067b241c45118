"""Matrix-free products J w, J' y and H v (MOI :JacVec / :HessVec) -- CPU side.

The generated product routines (rk4_dual_gen.h: ql_rk4_jvp_* / ql_rk4_vjp_* / ql_hess_prod_*) and the extra rows the
kernels add around them are emulated on the host with the kernels' headers (tests/native/emul_products.cpp).  The
emulation is checked bit for bit against the stated summation order (a left fold, in float64, of the emulated
SPARSE_TRUE and Hessian value streams), against the exact product of the oracle's matrices, and against the
extended-precision model's per-knot blocks.  The C ABI's argument checks and feature answers need no device."""
import ctypes as C
from fractions import Fraction

import numpy as np
import pytest

import quadruped_landing_b200 as ql
from quadruped_landing_b200 import evaluator as ev
from quadruped_landing_b200 import HybridNLP, build_problem, initial_guess
from oracle.oracle import Oracle

from conftest import _compile_native

# k_trans in {1, 2, N}, the jump at knot 1 and at knot N-1, pass boundaries (N = 33, 61, 129)
CLASSES = [(2, 1, 1), (2, 2, 2), (3, 2, 2), (33, 33, 1), (33, 1, 2), (61, 21, 1), (61, 21, 2), (129, 129, 2)]
EPS = np.finfo(np.float64).eps


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


@pytest.fixture(scope="session")
def prod_lib():
    L = C.CDLL(_compile_native("emul_products"))
    model = [C.c_int] * 3 + [C.c_double] * 4
    L.emul_jvp.argtypes = model + [C.c_void_p] * 3
    L.emul_vjp.argtypes = model + [C.c_void_p] * 3
    L.emul_hvp.argtypes = model + [C.c_void_p] * 5 + [C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]
    return L


def _point(prob, seed):
    rng = np.random.default_rng(seed)
    base = initial_guess(prob) if prob.k_trans > 1 else np.zeros(prob.n_nlp)
    Z = base + 5e-2 * rng.standard_normal(prob.n_nlp)
    Z[19::20] = np.clip(Z[19::20], 1e-3, 2e-2)
    Z[2::20] *= np.where(rng.random(prob.N) < 0.5, -1.0, 1.0)        # both branches of the body row (Q4)
    return Z


def _vectors(prob, seed):
    rng = np.random.default_rng(seed + 7)
    return (rng.standard_normal(prob.n_nlp), rng.standard_normal(prob.m_nlp), rng.standard_normal(prob.n_nlp),
            rng.standard_normal(prob.m_nlp), float(rng.uniform(0.3, 1.7)))


def fold_rows(rows, cols, vals, vec, nrows, transpose=False):
    """Left fold of vals * vec over the entries of each output row (J w: row r over ascending columns; transpose:
    column c over ascending rows), in float64 -- the order include/qlnlp.h states."""
    rows, cols = np.asarray(rows) - 1, np.asarray(cols) - 1
    out_idx, in_idx = (cols, rows) if transpose else (rows, cols)
    order = np.lexsort((in_idx, out_idx))
    acc = [None] * nrows
    for e in order.tolist():
        t = float(vals[e]) * float(vec[in_idx[e]])
        o = out_idx[e]
        acc[o] = t if acc[o] is None else acc[o] + t
    return np.array([np.nan if a is None else a for a in acc])


def mirrored(rows, cols, vals):
    off = rows != cols
    return (np.concatenate([rows, cols[off]]), np.concatenate([cols, rows[off]]), np.concatenate([vals, vals[off]]))


def exact_product(rows, cols, vals, vec, nout):
    """The exact product (rational arithmetic) and, per output, the number of terms and sum |a v|."""
    acc = [Fraction(0)] * nout
    mag = np.zeros(nout)
    cnt = np.zeros(nout)
    for r, c, a in zip((np.asarray(rows) - 1).tolist(), (np.asarray(cols) - 1).tolist(), np.asarray(vals).tolist()):
        acc[r] += Fraction(a) * Fraction(float(vec[c]))
        mag[r] += abs(a * vec[c])
        cnt[r] += 1
    return acc, cnt, mag


def assert_close_exact(got, exact, cnt, mag, extra=0.0, what=""):
    err = np.array([abs(float(Fraction(g) - e)) for g, e in zip(got.tolist(), exact)])
    tol = cnt * EPS * mag + 1e-14 + extra
    bad = np.nonzero(~(err <= tol))[0]
    assert not bad.size, (what, bad[:5].tolist(), err[bad[:5]].tolist(), tol[bad[:5]].tolist())


def _emul(prod_lib, emul_lib, prob, Z, w, y, v, lam, sigma):
    N, kt, im = prob.N, prob.k_trans, prob.init_mode
    m = prob.model
    args = (N, kt, im, m.g, m.mb, m.mf, m.lb)
    jw, jty, hv = np.empty(prob.m_nlp), np.empty(prob.n_nlp), np.empty(prob.n_nlp)
    assert prod_lib.emul_jvp(*args, Z.ctypes.data, w.ctypes.data, jw.ctypes.data) == 0
    assert prod_lib.emul_vjp(*args, Z.ctypes.data, y.ctypes.data, jty.ctypes.data) == 0
    assert prod_lib.emul_hvp(*args, prob.Q.ctypes.data, prob.R.ctypes.data, prob.q.ctypes.data, prob.r.ctypes.data,
                             Z.ctypes.data, sigma, lam.ctypes.data, v.ctypes.data, hv.ctypes.data) == 0
    nlp = HybridNLP.from_problem(prob, pattern="true")
    tvals = np.empty(nlp.nnz)
    assert emul_lib.emul_true_stream(*args, Z.ctypes.data, tvals.ctypes.data, nlp.nnz) == 0
    hvals = np.empty(nlp.nnz_hess)
    assert emul_lib.emul_hess_stream(*args, prob.Q.ctypes.data, prob.R.ctypes.data, prob.q.ctypes.data,
                                     prob.r.ctypes.data, Z.ctypes.data, sigma, lam.ctypes.data, hvals.ctypes.data,
                                     nlp.nnz_hess) == 0
    return nlp, jw, jty, hv, tvals, hvals


@pytest.mark.parametrize("N,kt,im", CLASSES)
def test_generated_products_are_the_fold_of_the_value_streams(prod_lib, emul_lib, N, kt, im):
    prob = build_problem(N=N, k_trans=kt, init_mode=im)
    for seed in range(2):
        Z = _point(prob, 10 * N + seed)
        w, y, v, lam, sigma = _vectors(prob, seed)
        nlp, jw, jty, hv, tvals, hvals = _emul(prod_lib, emul_lib, prob, Z, w, y, v, lam, sigma)
        rows, cols = nlp.jacobian_structure_arrays()
        assert np.array_equal(jw, fold_rows(rows, cols, tvals, w, prob.m_nlp))
        assert np.array_equal(jty, fold_rows(rows, cols, tvals, y, prob.n_nlp, transpose=True))
        hr, hc = nlp.hessian_structure_arrays()
        mr, mc, mv = mirrored(hr, hc, hvals)
        assert np.array_equal(hv, fold_rows(mr, mc, mv, v, prob.n_nlp))


@pytest.mark.parametrize("N,kt,im", CLASSES)
def test_products_against_the_exact_product_of_the_oracle_matrices(prod_lib, emul_lib, N, kt, im):
    prob = build_problem(N=N, k_trans=kt, init_mode=im)
    o = Oracle(prob)
    Z = _point(prob, 3 * N)
    w, y, v, lam, sigma = _vectors(prob, 1)
    nlp, jw, jty, hv, _, _ = _emul(prod_lib, emul_lib, prob, Z, w, y, v, lam, sigma)
    rows, cols = nlp.jacobian_structure_arrays()
    J = o.jac_c_dense(Z)
    vals = J[rows - 1, cols - 1]
    mask = np.zeros_like(J, dtype=bool)
    mask[rows - 1, cols - 1] = True
    assert not J[~mask].any()                           # the pattern holds every non-zero of the oracle's Jacobian
    assert_close_exact(jw, *exact_product(rows, cols, vals, w, prob.m_nlp), what="J w")
    assert_close_exact(jty, *exact_product(cols, rows, vals, y, prob.n_nlp), what="J' y")
    H = o.hess_lagrangian_dense(Z, sigma, lam)
    hr, hc = nlp.hessian_structure_arrays()
    mr, mc, _ = mirrored(hr, hc, np.zeros(len(hr)))
    hvals = H[mr - 1, mc - 1]
    # the generated second-order code matches the oracle's Hessian to 1e-12 of the block (test_hessian_cpu.py), not
    # bit for bit: allow that per entry on top of the rounding of the fold
    absv = np.zeros(prob.n_nlp)
    np.add.at(absv, mr - 1, np.abs(v[mc - 1]))
    assert_close_exact(hv, *exact_product(mr, mc, hvals, v, prob.n_nlp),
                       extra=1e-12 * max(1.0, np.abs(H).max()) * absv, what="H v")


@pytest.mark.parametrize("N,kt,im", [(33, 1, 2), (61, 21, 1), (129, 129, 2)])
def test_products_against_the_extended_precision_model(prod_lib, emul_lib, N, kt, im):
    """Per knot k of the sampled ones (pass boundaries, the jump, the end): (J' y) over knot k's columns is the model's
    block J_k' y[rows of k]; the defect rows of step k are J_k w_k + J_(k+1) w_(k+1); (H v) over knot k is H_k v_k."""
    pytest.importorskip("mpmath")
    from mp_nlp import Model, sample_knots
    prob = build_problem(N=N, k_trans=kt, init_mode=im)
    m = Model(prob)
    Z = _point(prob, 5 * N)
    w, y, v, lam, sigma = _vectors(prob, 2)
    _, jw, jty, hv, _, _ = _emul(prod_lib, emul_lib, prob, Z, w, y, v, lam, sigma)
    knots = sample_knots(N, kt)
    for k in knots:
        rows, Jk, _ = m.jac_knot(Z, k)
        nv = m.nvar(k)
        cs = slice(20 * (k - 1), 20 * (k - 1) + nv)
        want = Jk.T @ y[rows]
        tol = 1e-14 + 64 * EPS * (np.abs(Jk).T @ np.abs(y[rows]))
        assert np.all(np.abs(jty[cs] - want) <= tol), (k, np.abs(jty[cs] - want).max())
        if k < N:
            r1, J1, _ = m.jac_knot(Z, k + 1)
            dyn = np.arange(m.c_dyn + 15 * (k - 1), m.c_dyn + 15 * k)
            i0 = [rows.tolist().index(r) for r in dyn]
            i1 = [r1.tolist().index(r) for r in dyn]
            ns = slice(20 * k, 20 * k + m.nvar(k + 1))
            want = Jk[i0] @ w[cs] + J1[i1] @ w[ns]
            tol = 1e-14 + 64 * EPS * (np.abs(Jk[i0]) @ np.abs(w[cs]) + np.abs(J1[i1]) @ np.abs(w[ns]))
            assert np.all(np.abs(jw[dyn] - want) <= tol), (k, np.abs(jw[dyn] - want).max())
    for k in knots[:: max(1, len(knots) // 3)]:
        Hk = m.hess_knot(Z, k, sigma, lam)
        cs = slice(20 * (k - 1), 20 * (k - 1) + m.nvar(k))
        want = Hk @ v[cs]
        tol = 1e-14 + (1e-12 + 64 * EPS) * (np.abs(Hk) @ np.abs(v[cs])) + 1e-12 * np.abs(Hk).max() * np.abs(v[cs]).sum()
        assert np.all(np.abs(hv[cs] - want) <= tol), (k, np.abs(hv[cs] - want).max())


# ---- the C ABI without a device
def _ptr(a):
    return None if a is None else a.ctypes.data


def test_feature_answers_only_with_products():
    prob = build_problem(N=5, k_trans=3)
    assert HybridNLP.from_problem(prob).features_available() == ["Grad", "Jac"]
    assert HybridNLP.from_problem(prob, hessian=True).features_available() == ["Grad", "Jac", "Hess"]
    assert HybridNLP.from_problem(prob, products=True).features_available() == ["Grad", "Jac", "JacVec"]
    assert HybridNLP.from_problem(prob, products=True, hessian=True).features_available() == \
        ["Grad", "Jac", "Hess", "JacVec", "HessVec"]


def test_argument_checks_need_no_device():
    prob = build_problem(N=5, k_trans=3)
    nlp = HybridNLP.from_problem(prob)
    L = ql.load_library()
    n, m = nlp.n_nlp, nlp.m_nlp
    Z, w, jw, y, jty = np.zeros(n + 1), np.zeros(n + 1), np.zeros(m + 1), np.zeros(m + 1), np.zeros(n + 1)

    def jac(B, io_kw=None, pv_kw=None):
        io = ev._BatchIO()
        io.Z, io.ldz = Z.ctypes.data, n
        for k, val in (io_kw or {}).items():
            setattr(io, k, val)
        pv = ev._ProductIO(w.ctypes.data, n, jw.ctypes.data, m, y.ctypes.data, m, jty.ctypes.data, n)
        for k, val in (pv_kw or {}).items():
            setattr(pv, k, val)
        return L.qlnlp_eval_jacobian_products_batch_device(nlp._h, B, C.byref(io), C.byref(pv), None)

    assert jac(0, {"Z": None}, {"w": None, "y": None}) == ev.QLNLP_OK          # B = 0 before the pointer checks
    assert L.qlnlp_eval_jacobian_products_batch_device(nlp._h, 0, None, None, None) == ev.QLNLP_OK
    assert L.qlnlp_eval_jacobian_products_batch_device(nlp._h, 1, None, None, None) == ev.QLNLP_EINVAL
    assert jac(-1) == ev.QLNLP_EINVAL
    assert jac(1, {"Z": None}) == ev.QLNLP_EINVAL
    assert jac(1, {"jac": jw.ctypes.data, "ldjac": 10 ** 6}) == ev.QLNLP_EINVAL
    assert jac(1, pv_kw={"w": None, "y": None}) == ev.QLNLP_EINVAL
    assert jac(1, pv_kw={"jw": None}) == ev.QLNLP_EINVAL
    assert jac(1, pv_kw={"jty": None}) == ev.QLNLP_EINVAL
    assert jac(1, pv_kw={"w": None}) == ev.QLNLP_EINVAL                        # jw without w
    for short in ({"ldw": n - 1}, {"ldjw": m - 1}, {"ldy": m - 1}, {"ldjty": n - 1}):
        assert jac(2, pv_kw=short) == ev.QLNLP_EINVAL, short
    assert jac(2, {"ldz": n - 1}) == ev.QLNLP_EINVAL
    assert jac(2, {"g": y.ctypes.data, "ldg": m - 1}) == ev.QLNLP_EINVAL
    assert jac(2, {"grad": w.ctypes.data, "ldgrad": n - 1}) == ev.QLNLP_EINVAL
    assert "ld" in L.qlnlp_last_error().decode()

    lam, V, HV = np.zeros(m + 1), np.zeros(n + 1), np.zeros(n + 1)

    def hess(B, Zp=Z.ctypes.data, ldz=n, ldl=m, ldv=n, ldhv=n, lp=lam.ctypes.data, vp=V.ctypes.data, hp=HV.ctypes.data):
        return L.qlnlp_eval_hessian_product_batch_device(nlp._h, B, Zp, ldz, None, lp, ldl, vp, ldv, hp, ldhv, None)

    assert hess(0, Zp=None, lp=None, vp=None, hp=None) == ev.QLNLP_OK
    assert hess(-1) == ev.QLNLP_EINVAL
    for kw in ({"Zp": None}, {"lp": None}, {"vp": None}, {"hp": None}, {"ldz": n - 1}, {"ldl": m - 1}, {"ldv": n - 1},
               {"ldhv": n - 1}):
        assert hess(1, **kw) == ev.QLNLP_EINVAL, kw
    for fn in (L.qlnlp_eval_constraint_jacobian_product, L.qlnlp_eval_constraint_jacobian_transpose_product):
        assert fn(nlp._h, None, _ptr(w), _ptr(jw)) == ev.QLNLP_EINVAL
        assert fn(nlp._h, _ptr(Z), None, _ptr(jw)) == ev.QLNLP_EINVAL
        assert fn(nlp._h, _ptr(Z), _ptr(w), None) == ev.QLNLP_EINVAL
    assert L.qlnlp_eval_hessian_lagrangian_product(nlp._h, _ptr(Z), None, 1.0, _ptr(lam), _ptr(HV)) == ev.QLNLP_EINVAL
    assert L.qlnlp_eval_hessian_lagrangian_product(nlp._h, _ptr(Z), _ptr(V), 1.0, None, _ptr(HV)) == ev.QLNLP_EINVAL

    kin = HybridNLP.from_problem(prob, kinematics=True)
    assert L.qlnlp_eval_hessian_product_batch_device(kin._h, 1, _ptr(Z), n, None, _ptr(lam), m, _ptr(V), n, _ptr(HV), n,
                                                     None) == ev.QLNLP_EINVAL
    with pytest.raises(ev.QlnlpError, match="kinematic rows"):
        kin.eval_hessian_lagrangian_product(np.empty(n), Z[:n], V[:n], 1.0, np.zeros(kin.m_nlp))


@pytest.mark.skipif(_has_gpu(), reason="checks the no-GPU behaviour")
def test_callbacks_report_no_device():
    prob = build_problem(N=5, k_trans=3)
    nlp = HybridNLP.from_problem(prob, hessian=True, products=True)
    n, m = nlp.n_nlp, nlp.m_nlp
    x = initial_guess(prob)
    for call in (lambda: nlp.eval_constraint_jacobian_product(np.empty(m), x, np.ones(n)),
                 lambda: nlp.eval_constraint_jacobian_transpose_product(np.empty(n), x, np.ones(m)),
                 lambda: nlp.eval_hessian_lagrangian_product(np.empty(n), x, np.ones(n), 1.0, np.ones(m))):
        with pytest.raises(ev.QlnlpError) as e:
            call()
        assert e.value.code == ev.QLNLP_ENODEVICE
