"""KKT factor / factored solve (qlnlp_kkt_factor_batch_device, qlnlp_kkt_solve_factored_batch_device) -- CPU side: the
argument checks of both entry points, which run before any device work, and the factor size against the formula the
header documents."""
import ctypes as C

import numpy as np
import pytest

import quadruped_landing_b200 as ql
from quadruped_landing_b200 import evaluator as ev
from quadruped_landing_b200 import HybridNLP, build_problem


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def _ptr(a):
    return a.ctypes.data


def _size(N, nnz, m):
    return 4 + 210 * N + 300 * (N - 1) + nnz + m


@pytest.mark.parametrize("N,kt,im", [(2, 2, 1), (2, 1, 2), (5, 3, 1), (33, 21, 2), (61, 21, 1), (61, 21, 2),
                                     (1024, 1000, 1), (1024, 1, 2)])
def test_factor_size_is_the_documented_formula(N, kt, im):
    nlp = HybridNLP.from_problem(build_problem(N=N, k_trans=kt, init_mode=im), pattern="true")
    assert nlp.kkt_factor_size == _size(N, nlp.nnz, nlp.m_nlp)
    if (N, kt) == (61, 21):
        assert nlp.kkt_factor_size == 36747                 # the default instance, as include/qlnlp.h states


def test_argument_checks_need_no_device():
    prob = build_problem(N=5, k_trans=3)
    nlp = HybridNLP.from_problem(prob, pattern="true")
    L = ql.load_library()
    n, m, F = nlp.n_nlp, nlp.m_nlp, nlp.kkt_factor_size
    arrays = {name: np.zeros(w + 2) for name, w in (("hess", nlp.nnz_hess), ("jac", nlp.nnz), ("sx", n), ("dc", m),
                                                     ("factor", F), ("r1", n), ("r2", m), ("px", n), ("pl", m))}
    arrays["status"] = np.zeros(4, dtype=np.int32)
    arrays["index"] = np.zeros(4, dtype=np.int64)

    def fio(**kw):
        a = arrays
        io = ev._KktFactorIO(_ptr(a["hess"]), nlp.nnz_hess, _ptr(a["jac"]), nlp.nnz, _ptr(a["sx"]), n, _ptr(a["dc"]), m,
                             _ptr(a["factor"]), F, _ptr(a["status"]))
        for k, v in kw.items():
            setattr(io, k, v)
        return io

    def rio(**kw):
        a = arrays
        io = ev._KktRhsIO(_ptr(a["factor"]), F, 1, _ptr(a["index"]), _ptr(a["r1"]), n, _ptr(a["r2"]), m, _ptr(a["px"]), n,
                          _ptr(a["pl"]), m, _ptr(a["status"]))
        for k, v in kw.items():
            setattr(io, k, v)
        return io

    def factor(B, h=nlp, **kw):
        return L.qlnlp_kkt_factor_batch_device(h._h, B, C.byref(fio(**kw)), None)

    def solve(R, h=nlp, **kw):
        return L.qlnlp_kkt_solve_factored_batch_device(h._h, R, C.byref(rio(**kw)), None)

    # B = 0 / R = 0 before the pointer checks
    assert L.qlnlp_kkt_factor_batch_device(nlp._h, 0, None, None) == ev.QLNLP_OK
    assert L.qlnlp_kkt_solve_factored_batch_device(nlp._h, 0, None, None) == ev.QLNLP_OK
    assert factor(0, hess=None, factor=None, status=None) == ev.QLNLP_OK
    assert solve(0, factor=None, r1=None, status=None) == ev.QLNLP_OK
    assert L.qlnlp_kkt_factor_batch_device(nlp._h, 1, None, None) == ev.QLNLP_EINVAL
    assert L.qlnlp_kkt_solve_factored_batch_device(nlp._h, 1, None, None) == ev.QLNLP_EINVAL
    assert factor(-1) == ev.QLNLP_EINVAL and solve(-1) == ev.QLNLP_EINVAL
    assert solve(1, nfactor=-1) == ev.QLNLP_EINVAL
    # required pointers
    for name in ("hess", "jac", "dc", "factor", "status"):
        assert factor(1, **{name: None}) == ev.QLNLP_EINVAL, name
    for name in ("factor", "r1", "r2", "px", "pl", "status"):
        assert solve(1, **{name: None}) == ev.QLNLP_EINVAL, name
    # leading dimensions
    for name, w in (("ldhess", nlp.nnz_hess), ("ldjac", nlp.nnz), ("ldsx", n), ("lddc", m), ("ldfactor", F)):
        assert factor(2, **{name: w - 1}) == ev.QLNLP_EINVAL, name
        assert "ld" in L.qlnlp_last_error().decode()
    for name, w in (("ldfactor", F), ("ldr1", n), ("ldr2", m), ("ldpx", n), ("ldpl", m)):
        assert solve(2, **{name: w - 1}) == ev.QLNLP_EINVAL, name
        assert "ld" in L.qlnlp_last_error().decode()
    # alignment: 8 bytes, status 4
    for name in ("hess", "jac", "sx", "dc", "factor"):
        assert factor(1, **{name: _ptr(arrays[name]) + 4}) == ev.QLNLP_EINVAL, name
    assert factor(1, status=_ptr(arrays["status"]) + 2) == ev.QLNLP_EINVAL
    for name in ("factor", "index", "r1", "r2", "px", "pl"):
        assert solve(1, **{name: _ptr(arrays[name]) + 4}) == ev.QLNLP_EINVAL, name
    assert solve(1, status=_ptr(arrays["status"]) + 2) == ev.QLNLP_EINVAL

    # the handles the one-shot solve refuses, with its messages, whatever B; the size query refuses them too
    block = HybridNLP.from_problem(prob, pattern="block")
    dense = HybridNLP.from_problem(prob, use_sparse_jacobian=False)
    kin = HybridNLP.from_problem(prob, pattern="true", kinematics=True)
    multi = HybridNLP.from_problem(prob, pattern="true", devices=[0])
    out = C.c_int64()
    for h, what in ((block, "SPARSE_TRUE"), (dense, "SPARSE_TRUE"), (kin, "kinematic"), (multi, "multi-device")):
        for rc in (factor(1, h=h), factor(0, h=h), solve(1, h=h), solve(0, h=h),
                   L.qlnlp_kkt_factor_size(h._h, C.byref(out))):
            assert rc == ev.QLNLP_EINVAL
            assert what in L.qlnlp_last_error().decode()
        with pytest.raises(ql.QlnlpError):
            h.kkt_factor_size
    assert L.qlnlp_kkt_factor_size(nlp._h, None) == ev.QLNLP_EINVAL
    assert L.qlnlp_kkt_factor_size(None, C.byref(out)) == ev.QLNLP_EINVAL
    if not _has_gpu():
        # valid arguments reach the device
        assert factor(1) == ev.QLNLP_ENODEVICE
        assert factor(1, sx=None, ldsx=0) == ev.QLNLP_ENODEVICE                # sx is optional
        assert solve(1) == ev.QLNLP_ENODEVICE
        assert solve(3, index=None, nfactor=0) == ev.QLNLP_ENODEVICE           # index optional; rows beyond: status -2
