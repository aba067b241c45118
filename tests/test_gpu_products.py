"""Matrix-free products on the GPU (eval_prod_kernel, hess_prod_kernel): J w, J' y and H v equal, bit for bit, the
left fold of the GPU's own materialised values in the order include/qlnlp.h states, whatever the batch size, batch
position, leading dimensions, alignment, Jacobian pattern or entry point."""
import numpy as np
import pytest

import quadruped_landing_b200 as ql
from conftest import perturbed_batch
from oracle.oracle import Oracle
from test_products_cpu import assert_close_exact, exact_product, fold_rows, mirrored

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def _setup(N, kt, im, B, seed=0, **kw):
    p = ql.build_problem(N=N, k_trans=kt, init_mode=im)
    base = ql.initial_guess(p) if kt > 1 else np.zeros(p.n_nlp)
    Z = perturbed_batch(p, [base], B, 5e-2, seed)
    Z[:, 2::20] *= np.where(np.random.default_rng(seed).random((B, N)) < 0.5, -1.0, 1.0)     # both theta branches (Q4)
    return p, Z


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _np(t):
    torch.cuda.synchronize()
    return t.cpu().numpy()


def _dense_block(nlp, vals):
    rows, cols = nlp.jacobian_structure_arrays()
    J = np.zeros((nlp.m_nlp, nlp.n_nlp))
    J[rows - 1, cols - 1] = vals
    return J


def _sym_hessian(nlp, vals):
    rows, cols = nlp.hessian_structure_arrays()
    H = np.zeros((nlp.n_nlp, nlp.n_nlp))
    H[rows - 1, cols - 1] = vals
    H[cols - 1, rows - 1] = vals
    return H


@pytest.mark.parametrize("N,kt,im", [(2, 1, 1), (5, 3, 1), (33, 33, 1), (61, 21, 1), (61, 21, 2)])
def test_unit_vectors_rebuild_the_matrices(N, kt, im):
    p, Z1 = _setup(N, kt, im, 1, seed=N)
    nlp = ql.HybridNLP.from_problem(p, hessian=True, products=True)
    n, m = nlp.n_nlp, nlp.m_nlp
    J = _dense_block(nlp, _np(nlp.eval_batch(_cuda(Z1), want=("jac",))["jac"])[0])
    Zn, Zm = _cuda(np.repeat(Z1, n, axis=0)), _cuda(np.repeat(Z1, m, axis=0))
    jw = _np(nlp.eval_products_batch(Zn, w=_cuda(np.eye(n)))["jw"])
    assert np.array_equal(jw.T, J)                                        # column j of J = J e_j
    jty = _np(nlp.eval_products_batch(Zm, y=_cuda(np.eye(m)))["jty"])
    assert np.array_equal(jty, J)                                         # row i of J = J' e_i
    lam = np.random.default_rng(N).standard_normal((1, m))
    H = _sym_hessian(nlp, _np(nlp.eval_hessian_batch(_cuda(Z1), _cuda(lam)))[0])
    hv = _np(nlp.eval_hessian_product_batch(Zn, _cuda(np.repeat(lam, n, axis=0)), _cuda(np.eye(n))))
    assert np.array_equal(hv.T, H)


@pytest.mark.parametrize("ieee_div", [False, True])
@pytest.mark.parametrize("N,kt,im", [(61, 21, 1), (65, 2, 1), (129, 129, 2), (257, 100, 1), (1024, 1000, 1)])
def test_random_directions_are_the_fold_of_the_materialised_values(N, kt, im, ieee_div, monkeypatch):
    B = 6
    p, Z = _setup(N, kt, im, B, seed=3)
    monkeypatch.delenv("QLNLP_IEEE_DIV", raising=False)
    if ieee_div:
        monkeypatch.setenv("QLNLP_IEEE_DIV", "1")
    nlp = ql.HybridNLP.from_problem(p, pattern="true", hessian=True, products=True)
    monkeypatch.delenv("QLNLP_IEEE_DIV", raising=False)      # read once, when the handle is created
    rng = np.random.default_rng(N)
    w, y, v, lam = (rng.standard_normal((B, d)) for d in (nlp.n_nlp, nlp.m_nlp, nlp.n_nlp, nlp.m_nlp))
    sigma = rng.uniform(0.3, 1.7, B)
    Zd = _cuda(Z)
    out = nlp.eval_products_batch(Zd, w=_cuda(w), y=_cuda(y))
    hv = _np(nlp.eval_hessian_product_batch(Zd, _cuda(lam), _cuda(v), sigma=_cuda(sigma)))
    jw, jty = _np(out["jw"]), _np(out["jty"])
    vals = _np(nlp.eval_batch(Zd, want=("jac",))["jac"])
    hvals = _np(nlp.eval_hessian_batch(Zd, _cuda(lam), sigma=_cuda(sigma)))
    rows, cols = nlp.jacobian_structure_arrays()
    hr, hc = nlp.hessian_structure_arrays()
    for b in range(B):
        assert np.array_equal(jw[b], fold_rows(rows, cols, vals[b], w[b], nlp.m_nlp)), b
        assert np.array_equal(jty[b], fold_rows(rows, cols, vals[b], y[b], nlp.n_nlp, transpose=True)), b
        mr, mc, mv = mirrored(hr, hc, hvals[b])
        assert np.array_equal(hv[b], fold_rows(mr, mc, mv, v[b], nlp.n_nlp)), b
    # within rounding of the exact product of the oracle's matrices (first row)
    o = Oracle(p)
    ov = o.jac_c_sparse_true(Z[0])
    assert_close_exact(jw[0], *exact_product(rows, cols, ov, w[0], nlp.m_nlp), what="J w")
    assert_close_exact(jty[0], *exact_product(cols, rows, ov, y[0], nlp.n_nlp), what="J' y")
    if N <= 257:
        H = o.hess_lagrangian_dense(Z[0], sigma[0], lam[0])
        mr, mc, _ = mirrored(hr, hc, np.zeros(len(hr)))
        absv = np.zeros(nlp.n_nlp)
        np.add.at(absv, mr - 1, np.abs(v[0][mc - 1]))
        assert_close_exact(hv[0], *exact_product(mr, mc, H[mr - 1, mc - 1], v[0], nlp.n_nlp),
                           extra=1e-12 * max(1.0, np.abs(H).max()) * absv, what="H v")
    # and of the extended-precision model's blocks on pass boundaries, the jump and the end
    if N in (61, 1024):
        pytest.importorskip("mpmath")
        from mp_nlp import Model, sample_knots
        mdl = Model(p)
        eps = np.finfo(np.float64).eps
        for k in sample_knots(N, kt):
            r, Jk, _ = mdl.jac_knot(Z[0], k)
            cs = slice(20 * (k - 1), 20 * (k - 1) + mdl.nvar(k))
            err = np.abs(jty[0][cs] - Jk.T @ y[0][r])
            assert np.all(err <= 1e-14 + 64 * eps * (np.abs(Jk).T @ np.abs(y[0][r]))), k


def test_same_bits_everywhere():
    N, kt, im = 61, 21, 1
    B = 4096
    p, Z = _setup(N, kt, im, B, seed=11)
    nlp = ql.HybridNLP.from_problem(p, hessian=True, products=True)
    n, m = nlp.n_nlp, nlp.m_nlp
    rng = np.random.default_rng(5)
    w, y, v, lam = (rng.standard_normal((B, d)) for d in (n, m, n, m))
    Zd, wd, yd, vd, ld = _cuda(Z), _cuda(w), _cuda(y), _cuda(v), _cuda(lam)
    ref = nlp.eval_products_batch(Zd, w=wd, y=yd)
    jw, jty = _np(ref["jw"]), _np(ref["jty"])
    hv = _np(nlp.eval_hessian_product_batch(Zd, ld, vd))
    for Bs in (1, 7):                                                      # batch size, and batch position
        for lo in (0, 1000, B - Bs):
            s = slice(lo, lo + Bs)
            o = nlp.eval_products_batch(Zd[s], w=wd[s], y=yd[s])
            assert np.array_equal(_np(o["jw"]), jw[s]) and np.array_equal(_np(o["jty"]), jty[s])
            assert np.array_equal(_np(nlp.eval_hessian_product_batch(Zd[s], ld[s], vd[s])), hv[s])
    # the MOI callbacks
    for b in (0, 2345):
        a, t, h = np.empty(m), np.empty(n), np.empty(n)
        nlp.eval_constraint_jacobian_product(a, Z[b], w[b])
        nlp.eval_constraint_jacobian_transpose_product(t, Z[b], y[b])
        nlp.eval_hessian_lagrangian_product(h, Z[b], v[b], 1.0, lam[b])
        assert np.array_equal(a, jw[b]) and np.array_equal(t, jty[b]) and np.array_equal(h, hv[b])
    # every Jacobian pattern
    for kw in ({"pattern": "true"}, {"use_sparse_jacobian": False}):
        other = ql.HybridNLP.from_problem(p, **kw)
        o = other.eval_products_batch(Zd[:300], w=wd[:300], y=yd[:300])
        assert np.array_equal(_np(o["jw"]), jw[:300]) and np.array_equal(_np(o["jty"]), jty[:300])
    # odd leading dimensions and 8-byte (not 16-byte) aligned rows: plain loads and stores
    Bo = 333
    def odd(a, d):
        big = torch.zeros((Bo, d + 4), dtype=torch.float64, device="cuda")
        big[:, 1:1 + d] = a
        return big[:, 1:1 + d]
    outs = {"jw": odd(0, m), "jty": odd(0, n)}
    o = nlp.eval_products_batch(odd(Zd[:Bo], n), w=odd(wd[:Bo], n), y=odd(yd[:Bo], m), out=outs)
    assert np.array_equal(_np(o["jw"]), jw[:Bo]) and np.array_equal(_np(o["jty"]), jty[:Bo])
    h = nlp.eval_hessian_product_batch(odd(Zd[:Bo], n), odd(ld[:Bo], m), odd(vd[:Bo], n), out=odd(0, n))
    assert np.array_equal(_np(h), hv[:Bo])
    # interleaved with the evaluator and the Hessian on one stream (they share the stream's work counter)
    plain = nlp.eval_batch(Zd[:500])
    for _ in range(3):
        a = nlp.eval_products_batch(Zd, w=wd, y=yd)
        e = nlp.eval_batch(Zd[:500])
        hh = nlp.eval_hessian_batch(Zd[:200], ld[:200])
        c = nlp.eval_hessian_product_batch(Zd, ld, vd)
        assert np.array_equal(_np(a["jw"]), jw) and np.array_equal(_np(a["jty"]), jty)
        assert np.array_equal(_np(c), hv)
        for k in ("f", "grad", "g", "jac"):
            assert torch.equal(e[k], plain[k]), k
        assert np.array_equal(_np(hh), _np(nlp.eval_hessian_batch(Zd[:200], ld[:200])))


@pytest.mark.parametrize("with_x0xf", [False, True])
def test_fused_outputs_equal_eval_batch(with_x0xf):
    p, Z = _setup(61, 21, 2, 1000, seed=4)
    nlp = ql.HybridNLP.from_problem(p, products=True)
    rng = np.random.default_rng(9)
    kw = {}
    if with_x0xf:
        kw = {"x0": _cuda(p.x0 + 1e-2 * rng.standard_normal((1000, 15))), "xf": _cuda(p.xf + 1e-2 * rng.standard_normal((1000, 15)))}
    Zd = _cuda(Z)
    w, y = _cuda(rng.standard_normal((1000, nlp.n_nlp))), _cuda(rng.standard_normal((1000, nlp.m_nlp)))
    ref = nlp.eval_batch(Zd, want=("f", "grad", "g"), **kw)
    only = nlp.eval_products_batch(Zd, w=w, y=y)
    for want in (("f", "grad", "g"), ("g",), ("f",), ("grad",)):
        for vec in ({"w": w, "y": y}, {"w": w}, {"y": y}):
            o = nlp.eval_products_batch(Zd, want=want, **vec, **kw)
            for k in want:
                assert torch.equal(o[k], ref[k]), (want, k)
            for k in ("jw", "jty"):
                if k in o:
                    assert torch.equal(o[k], only[k]), k


def test_no_write_outside_the_rows():
    p, Z = _setup(61, 21, 1, 37, seed=5)
    nlp = ql.HybridNLP.from_problem(p, products=True)
    n, m = nlp.n_nlp, nlp.m_nlp
    B, guard, sentinel = 37, 3, -7.25
    rng = np.random.default_rng(1)
    Zd, wd, yd = _cuda(Z), _cuda(rng.standard_normal((B, n))), _cuda(rng.standard_normal((B, m)))
    ld = _cuda(rng.standard_normal((B, m)))
    for pad in (2, 3):
        big = {k: torch.full((B + 2 * guard, d + pad), sentinel, dtype=torch.float64, device="cuda")
               for k, d in (("jw", m), ("jty", n), ("hv", n))}
        views = {k: big[k][guard:guard + B, :d] for k, d in (("jw", m), ("jty", n), ("hv", n))}
        nlp.eval_products_batch(Zd, w=wd, y=yd, out={"jw": views["jw"], "jty": views["jty"]})
        nlp.eval_hessian_product_batch(Zd, ld, wd, out=views["hv"])
        torch.cuda.synchronize()
        for k, d in (("jw", m), ("jty", n), ("hv", n)):
            assert bool((big[k][:guard] == sentinel).all()) and bool((big[k][guard + B:] == sentinel).all()), k
            assert bool((big[k][:, d:] == sentinel).all()), k
            assert not bool((views[k] == sentinel).any()), k


@pytest.mark.parametrize("N,kt,im", [(61, 21, 1), (31, 11, 2), (2, 1, 1), (33, 33, 2), (65, 2, 1)])
def test_kinematic_rows(N, kt, im):
    B = 40
    p, Z = _setup(N, kt, im, B, seed=6)
    nlp = ql.HybridNLP.from_problem(p, pattern="true", kinematics=True, hessian=True, products=True)
    rng = np.random.default_rng(2)
    w, y = rng.standard_normal((B, nlp.n_nlp)), rng.standard_normal((B, nlp.m_nlp))
    Zd = _cuda(Z)
    ref = nlp.eval_batch(Zd, want=("g", "jac"))
    o = nlp.eval_products_batch(Zd, w=_cuda(w), y=_cuda(y), want=("g",))
    jw, jty, vals = _np(o["jw"]), _np(o["jty"]), _np(ref["jac"])
    assert torch.equal(o["g"], ref["g"])
    rows, cols = nlp.jacobian_structure_arrays()
    for b in range(B):
        assert np.array_equal(jw[b], fold_rows(rows, cols, vals[b], w[b], nlp.m_nlp)), b
        assert np.array_equal(jty[b], fold_rows(rows, cols, vals[b], y[b], nlp.n_nlp, transpose=True)), b
    a = np.empty(nlp.m_nlp)
    nlp.eval_constraint_jacobian_product(a, Z[1], w[1])
    assert np.array_equal(a, jw[1])
    with pytest.raises(ql.QlnlpError):
        nlp.eval_hessian_lagrangian_product(np.empty(nlp.n_nlp), Z[0], w[0], 1.0, y[0])


def test_multi_device_handle():
    p, Z = _setup(61, 21, 1, 8, seed=7)
    multi = ql.HybridNLP.from_problem(p, devices=[0], hessian=True, products=True)
    plain = ql.HybridNLP.from_problem(p, hessian=True, products=True)
    n, m = plain.n_nlp, plain.m_nlp
    rng = np.random.default_rng(3)
    w, y, v = rng.standard_normal(n), rng.standard_normal(m), rng.standard_normal(n)
    with pytest.raises(ql.QlnlpError, match="multi-device handle: the Jacobian products take a single-device handle"):
        multi.eval_products_batch(_cuda(Z), w=_cuda(np.tile(w, (8, 1))))
    with pytest.raises(ql.QlnlpError, match="multi-device handle: the Hessian takes a single-device handle"):
        multi.eval_hessian_product_batch(_cuda(Z), _cuda(np.tile(y, (8, 1))), _cuda(np.tile(v, (8, 1))))
    for nl in (multi, plain):
        a, t, h = np.empty(m), np.empty(n), np.empty(n)
        nl.eval_constraint_jacobian_product(a, Z[0], w)
        nl.eval_constraint_jacobian_transpose_product(t, Z[0], y)
        nl.eval_hessian_lagrangian_product(h, Z[0], v, 0.7, y)
        if nl is multi:
            got = (a, t, h)
        else:
            assert all(np.array_equal(g, r) for g, r in zip(got, (a, t, h)))
