"""Batched KKT solve on the GPU (kkt_kernel): the step solves the full sparse KKT system assembled on the CPU from the
handle's structures (tests/kkt_ref.py), the status is the inertia test, and the bits depend on the problem alone."""
import numpy as np
import pytest

import quadruped_landing_b200 as ql
from conftest import perturbed_batch
import kkt_ref

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _np(t):
    torch.cuda.synchronize()
    return t.cpu().numpy()


class Case:
    """B problems of one class with W and J from the device kernels at perturbed guesses and seeded multipliers.  The
    objective factor and the multipliers default to 1e-4: at sigma = 1 the x-h entries of the objective's Hessian (up to
    ~1e3 at the default costs) make W + diag(sx) + J' D^-1 J indefinite for these inputs, which the status test covers;
    at 1e-4, |W| <= 0.12 at N = 61 and M >= 0.9 I with sx in [1, 10]."""

    def __init__(self, N, kt, im, B, seed, Z=None, lam_scale=1e-4, sigma=None):
        sigma = np.full(B, 1e-4) if sigma is None else sigma
        self.p = ql.build_problem(N=N, k_trans=kt, init_mode=im)
        self.nlp = ql.HybridNLP.from_problem(self.p, pattern="true", hessian=True)
        nlp = self.nlp
        rng = np.random.default_rng(seed)
        if Z is None:
            base = ql.initial_guess(self.p) if kt > 1 else np.zeros(self.p.n_nlp)
            Z = perturbed_batch(self.p, [base], B, 5e-2, seed)
        self.Z = Z
        lam = lam_scale * rng.standard_normal((B, nlp.m_nlp))
        Zd = _cuda(Z)
        self.jac = nlp.eval_batch(Zd, want=("jac",))["jac"]
        self.hess = nlp.eval_hessian_batch(Zd, _cuda(lam), sigma=_cuda(sigma))
        self.hs, self.js = nlp.hessian_structure_arrays(), nlp.jacobian_structure_arrays()
        self.sx = rng.uniform(1.0, 10.0, (B, nlp.n_nlp))
        self.dc = rng.uniform(1e-2, 1.0, (B, nlp.m_nlp))
        self.r1 = rng.standard_normal((B, nlp.n_nlp))
        self.r2 = rng.standard_normal((B, nlp.m_nlp))

    def solve(self, **kw):
        args = dict(hess=self.hess, jac=self.jac, dc=_cuda(self.dc), r1=_cuda(self.r1), r2=_cuda(self.r2),
                    sx=_cuda(self.sx))
        args.update(kw)
        px, pl, st = self.nlp.kkt_solve_batch(**args)
        return _np(px), _np(pl), _np(st)

    def K(self, b, sx=None, dc=None):
        return kkt_ref.kkt_matrix(self.hs, _np(self.hess)[b], self.js, _np(self.jac)[b],
                                  self.sx[b] if sx is None else sx, self.dc[b] if dc is None else dc)


@pytest.mark.parametrize("N,kt,im", [(2, 2, 1), (2, 1, 2), (5, 3, 1), (33, 1, 2), (61, 21, 1), (61, 21, 2),
                                     (1024, 1000, 1)])
def test_step_solves_the_kkt_system(N, kt, im):
    """At Case's mild scalings (dc in [1e-2, 1], sx in [1, 10]), where the one-shot step's normwise backward error is
    1e-12 or better.  It is not at interior-point scalings: tests/test_gpu_kkt_accuracy.py has that envelope."""
    B = 3 if N > 100 else 8
    cs = Case(N, kt, im, B, seed=N + kt)
    px, pl, st = cs.solve()
    assert (st == 0).all()
    for b in range(B):
        K = cs.K(b)
        res, scale = kkt_ref.residual(K, px[b], pl[b], cs.r1[b], cs.r2[b])
        assert res <= 1e-12 * scale, (b, res, scale)
        if b < 2 and N <= 61:
            # forward error <= cond(K) x backward error (the dense condition number is formed up to N = 61; the
            # residual bound above is the check at longer horizons)
            qx, ql_ = kkt_ref.solve(K, cs.r1[b], cs.r2[b])
            z, zr = np.concatenate([px[b], pl[b]]), np.concatenate([qx, ql_])
            cond = np.linalg.cond(K.toarray())
            err = np.abs(z - zr).max() / np.abs(zr).max()
            print(f"N={N} kt={kt} im={im} b={b}: cond(K) {cond:.2e}, relative difference to spsolve {err:.2e}")
            assert err <= 1e-15 * cond, (b, cond, err)


def test_realistic_case_at_the_recorded_solutions(golden):
    """Z = the recorded solutions, dc = 1e-6 on the equality rows (1e-2 on the inequality rows), sx = 1: the
    quasi-definite KKT matrix of an interior-point iterate near convergence.  Observed on one B200 (1,000 W): relative
    residual ||K z - r||_inf / (||K||_inf ||z||_inf + ||r||_inf) between 3.9e-15 and 9.8e-15 over the six solutions, with
    ||K||_inf from 2.5e2 to 2.6e3 and cond(K) = 1.8e8 (solution 1); the bound is 1e-12 times max(1, cond(K) / 1e8)."""
    Z = np.stack([golden[f"data_{i}"] for i in range(1, 7)])
    cs = Case(61, 21, 1, 6, seed=5, Z=Z)
    lb, ub = cs.nlp.constraint_bounds()
    dc = np.where(lb == ub, 1e-6, 1e-2)
    cs.dc = np.tile(dc, (6, 1))
    cs.sx = np.full((6, cs.nlp.n_nlp), 1.0)
    px, pl, st = cs.solve()
    assert (st == 0).all()
    for b in range(6):
        K = cs.K(b)
        res, scale = kkt_ref.residual(K, px[b], pl[b], cs.r1[b], cs.r2[b])
        if b == 0:
            cond = np.linalg.cond(K.toarray())
        print(f"recorded solution {b + 1}: residual {res:.2e}, scale {scale:.2e}, relative {res / scale:.2e}, "
              f"||K||_inf {np.abs(K).sum(axis=1).max():.2e}, cond(K) {cond:.2e}")
        assert res <= 1e-12 * max(1.0, cond / 1e8) * scale, (b, res, scale, cond)


@pytest.mark.parametrize("N,kt,im", [(2, 2, 1), (5, 3, 1), (9, 4, 2)])
def test_status_is_the_inertia_test(N, kt, im):
    B = 24
    rng = np.random.default_rng(N)
    sigma = np.where(np.arange(B) % 2 == 0, 1e-4, -1.0)
    cs = Case(N, kt, im, B, seed=N, sigma=sigma)
    n = cs.nlp.n_nlp
    # even problems: sigma = 1e-4, sx in [1, 10], dc <= 1 -> M > 0; odd: sigma = -1, tiny sx, large dc -> indefinite
    cs.sx[1::2] = 1e-6 * rng.random((B // 2, n))
    cs.dc[1::2] *= 1e4
    px, pl, st = cs.solve()
    sides = set()
    for b in range(B):
        M = kkt_ref.schur_dense(cs.K(b), n)
        scale = np.abs(M).max()
        want = kkt_ref.status_of(M, N, tol=0.0)
        # only cases with a margin: the deciding leading block is clearly (in)definite
        k = want if want else N
        m = M[:20 * k - (5 if k == N else 0), :20 * k - (5 if k == N else 0)]
        if abs(np.linalg.eigvalsh(m).min()) < 1e-9 * scale:
            continue
        assert st[b] == want, (b, st[b], want)
        sides.add(want == 0)
        if want:
            assert np.isnan(px[b]).all() and np.isnan(pl[b]).all()
        else:
            assert np.isfinite(px[b]).all() and np.isfinite(pl[b]).all()
    assert sides == {True, False}
    # a dc entry <= 0 or not finite: status -1, whatever else the problem holds
    dc = cs.dc.copy()
    dc[0, 3], dc[2, -1], dc[4, 7] = 0.0, -1.0, np.nan
    px, pl, st = cs.solve(dc=_cuda(dc))
    assert st[0] == st[2] == st[4] == -1 and np.isnan(px[[0, 2, 4]]).all() and np.isnan(pl[[0, 2, 4]]).all()


def _placed(a, B, pos, ld, off, fill=np.nan, dtype=torch.float64):
    """a (one row) at row `pos` of a [B, ld] buffer, starting `off` doubles into the row; other rows random."""
    t = torch.full((B, ld + off), fill, dtype=dtype, device="cuda")
    rows = torch.randn((B, a.shape[-1]), dtype=dtype, device="cuda") if dtype == torch.float64 else None
    v = t[:, off:off + a.shape[-1]]
    if rows is not None:
        v.copy_(rows.abs() + 0.5)
    v[pos] = _cuda(a)
    return v


def test_bits_depend_on_the_problem_alone():
    cs = Case(61, 21, 1, 1, seed=11)
    nlp = cs.nlp
    one = dict(hess=_np(cs.hess)[0], jac=_np(cs.jac)[0], dc=cs.dc[0], r1=cs.r1[0], r2=cs.r2[0], sx=cs.sx[0])
    ref = None
    for B, pos, ld_extra, off in ((1, 0, 0, 0), (7, 3, 1, 0), (64, 63, 2, 1), (300, 150, 3, 1), (5000, 4097, 0, 1)):
        args = {k: _placed(v, B, pos, v.shape[-1] + ld_extra, off) for k, v in one.items()}
        for k in ("hess", "jac"):          # the rest of the batch: copies of the problem at their own positions
            args[k][:] = args[k][pos]
        args["dc"].clamp_(min=1e-2)
        n, m = nlp.n_nlp, nlp.m_nlp
        px = torch.full((B, n + ld_extra + off), 7.0, dtype=torch.float64, device="cuda")[:, off:off + n]
        pl = torch.full((B, m + ld_extra + off), 7.0, dtype=torch.float64, device="cuda")[:, off:off + m]
        st = torch.full((B,), 9, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            nlp.kkt_solve_batch(**args, out=(px, pl, st))
        side.synchronize()
        got = (_np(px)[pos], _np(pl)[pos], int(_np(st)[pos]))
        if ref is None:
            ref = got
        assert np.array_equal(got[0].view(np.int64), ref[0].view(np.int64)), (B, pos)
        assert np.array_equal(got[1].view(np.int64), ref[1].view(np.int64)), (B, pos)
        assert got[2] == ref[2] == 0


def test_no_write_outside_the_rows():
    cs = Case(33, 21, 2, 5, seed=2)
    n, m = cs.nlp.n_nlp, cs.nlp.m_nlp
    canary = 12345.678
    bufs = {}
    for name, w, dt in (("px", n, torch.float64), ("pl", m, torch.float64)):
        bufs[name] = torch.full((7, w + 3), canary, dtype=dt, device="cuda")
    st = torch.full((7,), 77, dtype=torch.int32, device="cuda")
    out = (bufs["px"][1:6, 1:1 + n], bufs["pl"][1:6, 1:1 + m], st[1:6])
    cs.solve(out=out)
    for name, w in (("px", n), ("pl", m)):
        a = _np(bufs[name])
        assert (a[0] == canary).all() and (a[6] == canary).all()
        assert (a[1:6, 0] == canary).all() and (a[1:6, 1 + w:] == canary).all()
        assert np.isfinite(a[1:6, 1:1 + w]).all() and not (a[1:6, 1:1 + w] == canary).any()
    s = _np(st)
    assert s[0] == 77 and s[6] == 77 and (s[1:6] == 0).all()


def test_pipeline_on_one_stream():
    """Evaluator (SPARSE_TRUE) -> Hessian -> KKT solve back to back on one stream, no host synchronise in between, on a
    C3-style batch (per-problem initial states of the drop-height x pitch sweep, device-built guesses)."""
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
        r1 = torch.randn((B, nlp.n_nlp), generator=gen, device="cuda", dtype=torch.float64)
        r2 = torch.randn((B, nlp.m_nlp), generator=gen, device="cuda", dtype=torch.float64)
        jac = nlp.eval_batch(Z, x0=x0d, want=("jac",))["jac"]
        hess = nlp.eval_hessian_batch(Z, lam, sigma=torch.full((B,), 1e-4, dtype=torch.float64, device="cuda"))
        px, pl, st = nlp.kkt_solve_batch(hess, jac, dc, r1, r2, sx=sx)
    s.synchronize()
    st = st.cpu().numpy()
    assert (st == 0).all()
    hs, js = nlp.hessian_structure_arrays(), nlp.jacobian_structure_arrays()
    for b in (0, 1, 2047, 4095):
        K = kkt_ref.kkt_matrix(hs, hess[b].cpu().numpy(), js, jac[b].cpu().numpy(), sx[b].cpu().numpy(),
                               dc[b].cpu().numpy())
        res, scale = kkt_ref.residual(K, px[b].cpu().numpy(), pl[b].cpu().numpy(), r1[b].cpu().numpy(),
                                      r2[b].cpu().numpy())
        assert res <= 1e-12 * scale, (b, res, scale)
