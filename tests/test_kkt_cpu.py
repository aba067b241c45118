"""Batched KKT solve (qlnlp_kkt_solve_batch_device) -- CPU side: the C ABI's argument checks, which run before any
device work, and the reference of tests/kkt_ref.py, checked against a dense solve and against the structure the kernel
relies on (M block tridiagonal, 15 non-zero rows in each off-diagonal block, M > 0 exactly when K has inertia (n, m, 0))."""
import ctypes as C

import numpy as np
import pytest

import quadruped_landing_b200 as ql
from quadruped_landing_b200 import evaluator as ev
from quadruped_landing_b200 import HybridNLP, build_problem

import kkt_ref


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def _ptr(a):
    return a.ctypes.data


def _io(nlp, arrays, **kw):
    n, m = nlp.n_nlp, nlp.m_nlp
    io = ev._KktIO(_ptr(arrays["hess"]), nlp.nnz_hess, _ptr(arrays["jac"]), nlp.nnz, _ptr(arrays["sx"]), n,
                   _ptr(arrays["dc"]), m, _ptr(arrays["r1"]), n, _ptr(arrays["r2"]), m, _ptr(arrays["px"]), n,
                   _ptr(arrays["pl"]), m, _ptr(arrays["status"]))
    for k, v in kw.items():
        setattr(io, k, v)
    return io


def test_argument_checks_need_no_device():
    prob = build_problem(N=5, k_trans=3)
    nlp = HybridNLP.from_problem(prob, pattern="true")
    L = ql.load_library()
    n, m = nlp.n_nlp, nlp.m_nlp
    arrays = {name: np.zeros(w + 2) for name, w in (("hess", nlp.nnz_hess), ("jac", nlp.nnz), ("sx", n), ("dc", m),
                                                     ("r1", n), ("r2", m), ("px", n), ("pl", m))}
    arrays["status"] = np.zeros(4, dtype=np.int32)

    def call(B, h=nlp, **kw):
        return L.qlnlp_kkt_solve_batch_device(h._h, B, C.byref(_io(nlp, arrays, **kw)), None)

    assert L.qlnlp_kkt_solve_batch_device(nlp._h, 0, None, None) == ev.QLNLP_OK       # B = 0 before the pointer checks
    assert call(0, hess=None, jac=None, status=None) == ev.QLNLP_OK
    assert L.qlnlp_kkt_solve_batch_device(nlp._h, 1, None, None) == ev.QLNLP_EINVAL
    assert call(-1) == ev.QLNLP_EINVAL
    for name in ("hess", "jac", "dc", "r1", "r2", "px", "pl", "status"):
        assert call(1, **{name: None}) == ev.QLNLP_EINVAL, name
    for name, w in (("ldhess", nlp.nnz_hess), ("ldjac", nlp.nnz), ("ldsx", n), ("lddc", m), ("ldr1", n), ("ldr2", m),
                    ("ldpx", n), ("ldpl", m)):
        assert call(2, **{name: w - 1}) == ev.QLNLP_EINVAL, name
        assert "ld" in L.qlnlp_last_error().decode()
    assert call(1, dc=_ptr(arrays["dc"]) + 4) == ev.QLNLP_EINVAL                      # misaligned
    assert call(1, status=_ptr(arrays["status"]) + 2) == ev.QLNLP_EINVAL

    block = HybridNLP.from_problem(prob, pattern="block")
    kin = HybridNLP.from_problem(prob, pattern="true", kinematics=True)
    multi = HybridNLP.from_problem(prob, pattern="true", devices=[0])
    for h, what in ((block, "SPARSE_TRUE"), (kin, "kinematic"), (multi, "multi-device")):
        assert call(1, h=h) == ev.QLNLP_EINVAL
        assert what in L.qlnlp_last_error().decode()
        assert call(0, h=h) == ev.QLNLP_EINVAL                                         # refused whatever B
    if not _has_gpu():
        assert call(1) == ev.QLNLP_ENODEVICE                                           # valid arguments reach the device
        assert call(1, sx=None, ldsx=0) == ev.QLNLP_ENODEVICE                          # sx is optional


def test_residual_argument_checks_need_no_device():
    """qlnlp_kkt_residual_batch_device: the solve's inputs plus px, pl in and s1, s2 out, each with its own leading
    dimension; the handles the KKT solve refuses are refused."""
    prob = build_problem(N=5, k_trans=3)
    nlp = HybridNLP.from_problem(prob, pattern="true")
    L = ql.load_library()
    n, m = nlp.n_nlp, nlp.m_nlp
    widths = (("hess", nlp.nnz_hess), ("jac", nlp.nnz), ("sx", n), ("dc", m), ("r1", n), ("r2", m), ("px", n), ("pl", m),
              ("s1", n), ("s2", m))
    arrays = {name: np.zeros(w + 2) for name, w in widths}

    def call(B, h=nlp, **kw):
        io = ev._KktResidualIO(*[v for name, w in widths for v in (_ptr(arrays[name]), w)])
        for k, v in kw.items():
            setattr(io, k, v)
        return L.qlnlp_kkt_residual_batch_device(h._h, B, C.byref(io), None)

    assert L.qlnlp_kkt_residual_batch_device(nlp._h, 0, None, None) == ev.QLNLP_OK
    assert L.qlnlp_kkt_residual_batch_device(nlp._h, 1, None, None) == ev.QLNLP_EINVAL
    assert call(-1) == ev.QLNLP_EINVAL
    for name in ("hess", "jac", "dc", "r1", "r2", "px", "pl", "s1", "s2"):
        assert call(1, **{name: None}) == ev.QLNLP_EINVAL, name
    for name, w in widths:
        assert call(2, **{"ld" + name: w - 1}) == ev.QLNLP_EINVAL, name
        assert "ld" + name in L.qlnlp_last_error().decode(), name
    for name, _ in widths:
        assert call(1, **{name: _ptr(arrays[name]) + 4}) == ev.QLNLP_EINVAL, name       # misaligned
    block = HybridNLP.from_problem(prob, pattern="block")
    dense = HybridNLP.from_problem(prob, use_sparse_jacobian=False)
    kin = HybridNLP.from_problem(prob, pattern="true", kinematics=True)
    multi = HybridNLP.from_problem(prob, pattern="true", devices=[0])
    for h, what in ((block, "SPARSE_TRUE"), (dense, "SPARSE_TRUE"), (kin, "kinematic"), (multi, "multi-device")):
        assert call(1, h=h) == ev.QLNLP_EINVAL
        assert what in L.qlnlp_last_error().decode()
        assert call(0, h=h) == ev.QLNLP_EINVAL
    if not _has_gpu():
        assert call(1) == ev.QLNLP_ENODEVICE
        assert call(1, sx=None, ldsx=0) == ev.QLNLP_ENODEVICE


def _random_problem(nlp, seed, sigma_scale=1.0):
    """W and J with random values on the handle's structures, and positive diagonals."""
    rng = np.random.default_rng(seed)
    hs, js = nlp.hessian_structure_arrays(), nlp.jacobian_structure_arrays()
    hv = sigma_scale * rng.standard_normal(nlp.nnz_hess)
    jv = rng.standard_normal(nlp.nnz)
    sx = rng.uniform(1.0, 10.0, nlp.n_nlp)
    dc = rng.uniform(1e-2, 1.0, nlp.m_nlp)
    return hs, hv, js, jv, sx, dc, rng.standard_normal(nlp.n_nlp), rng.standard_normal(nlp.m_nlp)


@pytest.mark.parametrize("N,kt,im", [(2, 2, 1), (2, 1, 2), (5, 3, 1), (9, 4, 2), (12, 12, 1)])
def test_reference_matches_a_dense_solve(N, kt, im):
    nlp = HybridNLP.from_problem(build_problem(N=N, k_trans=kt, init_mode=im), pattern="true")
    hs, hv, js, jv, sx, dc, r1, r2 = _random_problem(nlp, N * 10 + kt)
    K = kkt_ref.kkt_matrix(hs, hv, js, jv, sx, dc)
    px, pl = kkt_ref.solve(K, r1, r2)
    z = np.linalg.solve(K.toarray(), np.concatenate([r1, r2]))
    cond = np.linalg.cond(K.toarray())
    assert np.abs(np.concatenate([px, pl]) - z).max() <= 1e-14 * cond * np.abs(z).max()
    res, scale = kkt_ref.residual(K, px, pl, r1, r2)
    assert res <= 1e-12 * scale
    # the eliminated form the kernel solves gives the same step
    n = nlp.n_nlp
    M = kkt_ref.schur_dense(K, n)
    Jd = K[n:, :n].toarray()
    px2 = np.linalg.solve(M, r1 + Jd.T @ (r2 / dc))
    assert np.abs(px2 - px).max() <= 1e-14 * np.linalg.cond(M) * np.abs(px).max()
    assert np.abs((Jd @ px2 - r2) / dc - pl).max() <= 1e-14 * cond * np.abs(pl).max()


@pytest.mark.parametrize("N,kt,im", [(2, 2, 1), (5, 3, 1), (9, 1, 2), (33, 21, 1)])
def test_eliminated_matrix_is_block_tridiagonal(N, kt, im):
    nlp = HybridNLP.from_problem(build_problem(N=N, k_trans=kt, init_mode=im), pattern="true")
    hs, hv, js, jv, sx, dc, _, _ = _random_problem(nlp, N)
    M = kkt_ref.schur_dense(kkt_ref.kkt_matrix(hs, hv, js, jv, sx, dc), nlp.n_nlp)
    knot = np.arange(nlp.n_nlp) // 20
    far = np.abs(knot[:, None] - knot[None, :]) > 1
    assert not M[far].any()
    for k in range(N - 1):                        # block (k+1, k): only the 15 state rows of knot k+1 are non-zero
        blk = M[20 * (k + 1):20 * (k + 1) + 20, 20 * k:20 * k + 20]
        assert not blk[15:].any() and blk[:15].any()


@pytest.mark.parametrize("N,kt,im", [(2, 2, 1), (5, 3, 1), (9, 4, 2)])
def test_positive_definite_eliminated_matrix_is_the_inertia_test(N, kt, im):
    """Haynsworth: with dc > 0, M > 0 exactly when K has n positive and m negative eigenvalues."""
    nlp = HybridNLP.from_problem(build_problem(N=N, k_trans=kt, init_mode=im), pattern="true")
    n, m = nlp.n_nlp, nlp.m_nlp
    seen = set()
    for seed in range(12):
        scale = [0.1, 3.0, 30.0][seed % 3]
        hs, hv, js, jv, sx, dc, _, _ = _random_problem(nlp, 100 + seed, sigma_scale=scale)
        dc = dc * (1.0 if seed % 2 else 100.0)
        K = kkt_ref.kkt_matrix(hs, hv, js, jv, sx, dc)
        ev_k = np.linalg.eigvalsh(K.toarray())
        pd = np.linalg.eigvalsh(kkt_ref.schur_dense(K, n)).min() > 0
        assert pd == ((ev_k > 0).sum() == n and (ev_k < 0).sum() == m)
        seen.add(pd)
    assert seen == {True, False}
