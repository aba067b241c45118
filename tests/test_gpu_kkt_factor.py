"""KKT factor / factored solve on the GPU (kkt_factor_kernel, kkt_solve_factored_kernel): a factor followed by a
factored solve gives the bits of the one-shot solve (kkt_kernel), many right-hand sides share one factor through
`index`, a factor is self-contained, and the bits depend on the problem alone."""
import numpy as np
import pytest

import quadruped_landing_b200 as ql
from quadruped_landing_b200 import evaluator as qev
import kkt_ref
from test_gpu_kkt import Case, _cuda, _np, _placed

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def _same_bits(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.int64), np.ascontiguousarray(b).view(np.int64))


def _factor(cs, dc=None, sx=True):
    return cs.nlp.kkt_factor_batch(cs.hess, cs.jac, _cuda(cs.dc if dc is None else dc), sx=_cuda(cs.sx) if sx else None)


def _solve(cs, factor, r1=None, r2=None, index=None):
    r1 = cs.r1 if r1 is None else r1
    r2 = cs.r2 if r2 is None else r2
    idx = None if index is None else torch.as_tensor(np.asarray(index, dtype=np.int64), device="cuda")
    px, pl, st = cs.nlp.kkt_solve_factored_batch(factor, _cuda(r1), _cuda(r2), index=idx)
    return _np(px), _np(pl), _np(st)


def _assert_same(got, want, what=""):
    assert _same_bits(got[0], want[0]), what
    assert _same_bits(got[1], want[1]), what
    assert np.array_equal(got[2], want[2]), (what, got[2], want[2])


@pytest.mark.parametrize("N,kt,im", [(2, 2, 1), (2, 1, 2), (5, 3, 1), (5, 3, 2), (33, 21, 1), (33, 1, 2), (61, 21, 1),
                                     (61, 21, 2), (1024, 1000, 1), (1024, 1000, 2)])
def test_factored_solve_gives_the_one_shot_bits(N, kt, im):
    B = 3 if N > 100 else 8
    cs = Case(N, kt, im, B, seed=N + kt + im)
    want = cs.solve()
    factor, fst = _factor(cs)
    assert factor.shape == (B, cs.nlp.kkt_factor_size)
    assert np.array_equal(_np(fst), want[2])
    _assert_same(_solve(cs, factor), want, (N, kt, im))
    # without sx
    want = cs.solve(sx=None)
    _assert_same(_solve(cs, _factor(cs, sx=False)[0]), want, "sx = 0")


@pytest.mark.parametrize("N,kt,im", [(2, 2, 1), (5, 3, 1), (9, 4, 2)])
def test_status_and_nan_rows_are_the_one_shot_ones(N, kt, im):
    """The inputs of test_gpu_kkt.py::test_status_is_the_inertia_test: half the problems indefinite, then dc <= 0."""
    B = 24
    rng = np.random.default_rng(N)
    sigma = np.where(np.arange(B) % 2 == 0, 1e-4, -1.0)
    cs = Case(N, kt, im, B, seed=N, sigma=sigma)
    cs.sx[1::2] = 1e-6 * rng.random((B // 2, cs.nlp.n_nlp))
    cs.dc[1::2] *= 1e4
    want = cs.solve()
    factor, fst = _factor(cs)
    got = _solve(cs, factor)
    _assert_same(got, want)
    assert np.array_equal(_np(fst), want[2])
    assert (want[2] == 0).any() and (want[2] > 0).any()
    dc = cs.dc.copy()
    dc[0, 3], dc[2, -1], dc[4, 7] = 0.0, -1.0, np.nan
    want = cs.solve(dc=_cuda(dc))
    factor, fst = _factor(cs, dc=dc)
    _assert_same(_solve(cs, factor), want)
    assert want[2][0] == want[2][2] == want[2][4] == -1 and np.array_equal(_np(fst), want[2])


def test_many_right_hand_sides_share_a_factor():
    B, per = 6, 5
    cs = Case(61, 21, 1, B, seed=3)
    nlp = cs.nlp
    rng = np.random.default_rng(7)
    factor, _ = _factor(cs)
    hess, jac = _np(cs.hess), _np(cs.jac)

    def one_shot(index, r1, r2):
        return cs.solve(hess=_cuda(hess[index]), jac=_cuda(jac[index]), dc=_cuda(cs.dc[index]), sx=_cuda(cs.sx[index]),
                        r1=_cuda(r1), r2=_cuda(r2))

    for name, index in (("five per factor", np.repeat(np.arange(B), per)),
                        ("permuted", rng.permutation(np.repeat(np.arange(B), 2))),
                        ("repeated", np.zeros(7, dtype=np.int64)),
                        ("subset", np.array([4, 1]))):
        R = len(index)
        r1 = rng.standard_normal((R, nlp.n_nlp))
        r2 = rng.standard_normal((R, nlp.m_nlp))
        got = _solve(cs, factor, r1, r2, index)
        assert (got[2] == 0).all(), name
        _assert_same(got, one_shot(index, r1, r2), name)
        for i in range(0, R, max(1, R // 4)):
            b = index[i]
            K = kkt_ref.kkt_matrix(cs.hs, hess[b], cs.js, jac[b], cs.sx[b], cs.dc[b])
            res, scale = kkt_ref.residual(K, got[0][i], got[1][i], r1[i], r2[i])
            assert res <= 1e-12 * scale, (name, i, res, scale)
    # without index: row i uses factor i, and rows beyond the factors are out of range
    r1 = rng.standard_normal((B + 2, nlp.n_nlp))
    r2 = rng.standard_normal((B + 2, nlp.m_nlp))
    got = _solve(cs, factor, r1, r2)
    assert np.array_equal(got[2], [0] * B + [-2, -2])
    _assert_same(tuple(g[:B] for g in got), one_shot(np.arange(B), r1[:B], r2[:B]), "no index")
    # an index outside [0, B): status -2 and NaN rows, the other rows untouched by it
    index = np.array([-1, B, 2, 1 << 40])
    got = _solve(cs, factor, r1[:4], r2[:4], index)
    assert np.array_equal(got[2], [-2, -2, 0, -2])
    assert np.isnan(got[0][[0, 1, 3]]).all() and np.isnan(got[1][[0, 1, 3]]).all()
    _assert_same(tuple(g[2:3] for g in got), one_shot(index[2:3], r1[2:3], r2[2:3]), "beside bad rows")
    # a factor of another class (same sizes, other initial mode): -3 on this handle
    other = ql.HybridNLP.from_problem(ql.build_problem(N=61, k_trans=21, init_mode=2), pattern="true")
    assert other.kkt_factor_size == nlp.kkt_factor_size
    px, pl, st = other.kkt_solve_factored_batch(factor, _cuda(r1[:B]), _cuda(r2[:B]))
    assert (_np(st) == -3).all() and torch.isnan(px).all() and torch.isnan(pl).all()


def test_factor_is_self_contained():
    cs = Case(33, 21, 2, 5, seed=4)
    hess, jac, dc, sx = cs.hess, cs.jac, _cuda(cs.dc), _cuda(cs.sx)
    factor, _ = cs.nlp.kkt_factor_batch(hess, jac, dc, sx=sx)
    before = _solve(cs, factor)
    assert (before[2] == 0).all()
    for t in (hess, jac, dc, sx):
        t.copy_(torch.rand_like(t) - 0.5)
    _assert_same(_solve(cs, factor), before, "inputs overwritten")


def test_bits_depend_on_the_problem_alone():
    cs = Case(61, 21, 1, 1, seed=11)
    nlp = cs.nlp
    n, m, size = nlp.n_nlp, nlp.m_nlp, nlp.kkt_factor_size
    inp = dict(hess=_np(cs.hess)[0], jac=_np(cs.jac)[0], dc=cs.dc[0], sx=cs.sx[0])
    rhs = dict(r1=cs.r1[0], r2=cs.r2[0])
    ref = cs.solve()
    for B, pos, ld_extra, off in ((1, 0, 0, 0), (7, 3, 1, 0), (64, 63, 2, 1), (300, 150, 3, 1), (2000, 1597, 0, 1)):
        args = {k: _placed(v, B, pos, v.shape[-1] + ld_extra, off) for k, v in inp.items()}
        for k in ("hess", "jac"):
            args[k][:] = args[k][pos]
        args["dc"].clamp_(min=1e-2)
        fac = torch.full((B, size + ld_extra + off), 7.0, dtype=torch.float64, device="cuda")[:, off:off + size]
        fst = torch.full((B,), 9, dtype=torch.int32, device="cuda")
        R = B + 3                             # right-hand sides at their own positions, factor row through index
        r = {k: _placed(v, R, R - 1 - pos, v.shape[-1] + ld_extra, off) for k, v in rhs.items()}
        index = torch.randint(0, B, (R,), dtype=torch.int64, device="cuda")
        index[R - 1 - pos] = pos
        px = torch.full((R, n + ld_extra + off), 7.0, dtype=torch.float64, device="cuda")[:, off:off + n]
        pl = torch.full((R, m + ld_extra + off), 7.0, dtype=torch.float64, device="cuda")[:, off:off + m]
        st = torch.full((R,), 9, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            nlp.kkt_factor_batch(args["hess"], args["jac"], args["dc"], sx=args["sx"], out=(fac, fst))
            nlp.kkt_solve_factored_batch(fac, r["r1"], r["r2"], index=index, out=(px, pl, st))
        side.synchronize()
        i = R - 1 - pos
        got = (_np(px)[i:i + 1], _np(pl)[i:i + 1], _np(st)[i:i + 1])
        _assert_same(got, ref, (B, pos))


def test_no_write_outside_the_rows():
    cs = Case(33, 21, 2, 5, seed=2)
    n, m, size = cs.nlp.n_nlp, cs.nlp.m_nlp, cs.nlp.kkt_factor_size
    canary = 12345.678
    fbuf = torch.full((7, size + 3), canary, dtype=torch.float64, device="cuda")
    fst = torch.full((7,), 77, dtype=torch.int32, device="cuda")
    factor, _ = cs.nlp.kkt_factor_batch(cs.hess, cs.jac, _cuda(cs.dc), sx=_cuda(cs.sx),
                                        out=(fbuf[1:6, 1:1 + size], fst[1:6]))
    bufs = {name: torch.full((7, w + 3), canary, dtype=torch.float64, device="cuda") for name, w in (("px", n), ("pl", m))}
    st = torch.full((7,), 77, dtype=torch.int32, device="cuda")
    cs.nlp.kkt_solve_factored_batch(factor, _cuda(cs.r1), _cuda(cs.r2),
                                    out=(bufs["px"][1:6, 1:1 + n], bufs["pl"][1:6, 1:1 + m], st[1:6]))
    for name, w in (("factor", size), ("px", n), ("pl", m)):
        a = _np(fbuf if name == "factor" else bufs[name])
        assert (a[0] == canary).all() and (a[6] == canary).all(), name
        assert (a[1:6, 0] == canary).all() and (a[1:6, 1 + w:] == canary).all(), name     # padding beyond the size
        if name != "factor":
            assert np.isfinite(a[1:6, 1:1 + w]).all() and not (a[1:6, 1:1 + w] == canary).any()
    for s in (_np(fst), _np(st)):
        assert s[0] == 77 and s[6] == 77 and (s[1:6] == 0).all()


def _refused_in_capture(call):
    x = torch.zeros(4, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    err = None
    with torch.cuda.graph(g):
        x.add_(1.0)
        try:
            call()
        except ql.QlnlpError as e:
            err = e
    assert err is not None and err.code == qev.QLNLP_EINVAL, str(err)
    assert "warm the handle" in str(err), str(err)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(x, torch.ones_like(x))


def test_streams_and_graphs():
    B = 64
    cs = Case(61, 21, 1, B, seed=9)
    nlp, n, m, size = cs.nlp, cs.nlp.n_nlp, cs.nlp.m_nlp, cs.nlp.kkt_factor_size
    dc, sx, r1, r2 = _cuda(cs.dc), _cuda(cs.sx), _cuda(cs.r1), _cuda(cs.r2)
    q1, q2 = torch.flip(r1, [0]).contiguous(), torch.flip(r2, [0]).contiguous()
    # a first factor or factored solve inside a capture is refused (the tables are not set up), the capture survives
    fresh = ql.HybridNLP.from_problem(cs.p, pattern="true")
    fresh.eval_batch(_cuda(cs.Z[:2]), want=("g",))
    torch.cuda.synchronize()
    _refused_in_capture(lambda: fresh.kkt_factor_batch(cs.hess, cs.jac, dc, sx=sx))
    fresh2 = ql.HybridNLP.from_problem(cs.p, pattern="true")
    fresh2.eval_batch(_cuda(cs.Z[:2]), want=("g",))
    torch.cuda.synchronize()
    fac0 = torch.zeros((1, size), dtype=torch.float64, device="cuda")
    _refused_in_capture(lambda: fresh2.kkt_solve_factored_batch(fac0, r1[:1], r2[:1]))
    # eager reference bits (this warms the handle)
    fac, fst = nlp.kkt_factor_batch(cs.hess, cs.jac, dc, sx=sx)
    want1 = nlp.kkt_solve_factored_batch(fac, r1, r2)
    want2 = nlp.kkt_solve_factored_batch(fac, q1, q2)
    assert _same_bits(_np(want1[0]), cs.solve()[0])
    want = [t.clone() for t in (fac, fst, *want1, *want2)]
    # captured factor -> solve -> solve, replayed beside eager launches on other streams
    outs = [torch.empty_like(t) for t in want]
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        nlp.kkt_factor_batch(cs.hess, cs.jac, dc, sx=sx, out=(outs[0], outs[1]))
        nlp.kkt_solve_factored_batch(outs[0], r1, r2, out=tuple(outs[2:5]))
        nlp.kkt_solve_factored_batch(outs[0], q1, q2, out=tuple(outs[5:8]))
    side = [torch.cuda.Stream() for _ in range(2)]
    eager = [[torch.empty_like(t) for t in want] for _ in side]
    for rep in range(3):
        for o in outs + [t for e in eager for t in e]:
            o.fill_(float("nan")) if o.dtype == torch.float64 else o.fill_(-9)
        torch.cuda.synchronize()
        g.replay()
        for s, e in zip(side, eager):
            with torch.cuda.stream(s):
                nlp.kkt_factor_batch(cs.hess, cs.jac, dc, sx=sx, out=(e[0], e[1]))
                nlp.kkt_solve_factored_batch(e[0], r1, r2, out=tuple(e[2:5]))
                nlp.kkt_solve_factored_batch(e[0], q1, q2, out=tuple(e[5:8]))
        torch.cuda.synchronize()
        for got in [outs] + eager:
            for a, b in zip(got, want):
                assert _same_bits(_np(a), _np(b)), rep


def test_pipeline_on_one_stream():
    """Evaluator (SPARSE_TRUE) -> Hessian -> factor -> two factored solves back to back on one stream, no host
    synchronise in between, on the C3-style batch of test_gpu_kkt.py::test_pipeline_on_one_stream."""
    p = ql.default_problem()
    nlp = ql.HybridNLP.from_problem(p, pattern="true", hessian=True)
    B = 4096
    x0 = ql.sweep_initial_states(p.model, np.linspace(0.25, 3.0, 64), np.linspace(-40.0, -5.0, 64))
    gen = torch.Generator(device="cuda").manual_seed(1)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        x0d = _cuda(x0)
        Z = nlp.initial_guess_batch(x0d)
        Z.add_(1e-3 * torch.randn(Z.shape, generator=gen, device="cuda", dtype=torch.float64))
        lam = 1e-4 * torch.randn((B, nlp.m_nlp), generator=gen, device="cuda", dtype=torch.float64)
        dc = 1e-2 + torch.rand((B, nlp.m_nlp), generator=gen, device="cuda", dtype=torch.float64)
        sx = 1.0 + 9.0 * torch.rand((B, nlp.n_nlp), generator=gen, device="cuda", dtype=torch.float64)
        r1 = torch.randn((2 * B, nlp.n_nlp), generator=gen, device="cuda", dtype=torch.float64)
        r2 = torch.randn((2 * B, nlp.m_nlp), generator=gen, device="cuda", dtype=torch.float64)
        jac = nlp.eval_batch(Z, x0=x0d, want=("jac",))["jac"]
        hess = nlp.eval_hessian_batch(Z, lam, sigma=torch.full((B,), 1e-4, dtype=torch.float64, device="cuda"))
        fac, fst = nlp.kkt_factor_batch(hess, jac, dc, sx=sx)
        a = nlp.kkt_solve_factored_batch(fac, r1[:B], r2[:B])
        index = torch.arange(B, dtype=torch.int64, device="cuda").flip(0)
        b = nlp.kkt_solve_factored_batch(fac, r1[B:], r2[B:], index=index)
        one = nlp.kkt_solve_batch(hess, jac, dc, r1[:B], r2[:B], sx=sx)
    s.synchronize()
    assert (fst.cpu().numpy() == 0).all() and (a[2].cpu().numpy() == 0).all() and (b[2].cpu().numpy() == 0).all()
    for x, y in zip(a, one):
        assert torch.equal(x, y)
    hs, js = nlp.hessian_structure_arrays(), nlp.jacobian_structure_arrays()
    npy = lambda t: t.cpu().numpy()
    for i in (0, 1, 2047, 4095):
        for sol, row, rr in ((a, i, i), (b, B - 1 - i, B + i)):
            K = kkt_ref.kkt_matrix(hs, npy(hess[row]), js, npy(jac[row]), npy(sx[row]), npy(dc[row]))
            res, scale = kkt_ref.residual(K, npy(sol[0][i]), npy(sol[1][i]), npy(r1[rr]), npy(r2[rr]))
            assert res <= 1e-12 * scale, (i, res, scale)
