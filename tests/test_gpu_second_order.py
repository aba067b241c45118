"""The second-order kernels (hess_kernel, hess_prod_kernel, eval_prod_kernel, kkt_kernel) at the inputs their other
tests skip: the IEEE-division instantiations against the reciprocal-FMA ones, the products at theta = 0 exactly, the
KKT solve without sx and with failures planted at known knots, and non-finite or failing problems mixed into batches
long enough that every resident warp takes several problems in turn."""
import os

import numpy as np
import pytest

import quadruped_landing_b200 as ql
from conftest import perturbed_batch
import kkt_ref
from test_mp_reference_cpu import random_problem, theta_edges
from test_products_cpu import fold_rows, mirrored
from test_second_order_cpu import planted_entry, planted_value, spd_w

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

EPS = np.finfo(np.float64).eps
F64 = torch.float64


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _np(t):
    torch.cuda.synchronize()
    return t.cpu().numpy()


def _handle(p, ieee_div, **kw):
    """A handle of ``p``; with ieee_div, created under QLNLP_IEEE_DIV (read once, when the handle is created)."""
    old = os.environ.pop("QLNLP_IEEE_DIV", None)
    try:
        if ieee_div:
            os.environ["QLNLP_IEEE_DIV"] = "1"
        return ql.HybridNLP.from_problem(p, **kw)
    finally:
        os.environ.pop("QLNLP_IEEE_DIV", None)
        if old is not None:
            os.environ["QLNLP_IEEE_DIV"] = old


def _same_bits(a, b):
    return torch.equal(a.contiguous().view(torch.int64), b.contiguous().view(torch.int64))


# ---- A. division instantiations

@pytest.mark.parametrize("which", ["default", "random-1", "random-2"])
def test_division_instantiations_agree(which):
    """For finite operands of ordinary magnitude both divisions return the correctly rounded quotient, so the FASTDIV
    and IEEE-division kernels must give the same numbers (sign of zero aside).  The default problem, and random model
    constants and cost tables in both initial modes."""
    p = ql.default_problem() if which == "default" else random_problem(23, im=int(which[-1]))
    B = 300
    Z = perturbed_batch(p, [ql.initial_guess(p)], B, 5e-2, 7)
    rng = np.random.default_rng(8)
    Z[:, 2::20] *= np.where(rng.random((B, p.N)) < 0.5, -1.0, 1.0)              # both theta branches (Q4)
    n, m = p.n_nlp, p.m_nlp
    Zd, lam, v, w, y = _cuda(Z), *(_cuda(rng.standard_normal((B, d))) for d in (m, n, n, m))
    sigma = _cuda(rng.uniform(0.3, 1.7, B))
    outs = []
    for ieee in (False, True):
        nlp = _handle(p, ieee, pattern="true", hessian=True, products=True)
        o = nlp.eval_products_batch(Zd, w=w, y=y, want=("f", "grad", "g"))
        o["hess"] = nlp.eval_hessian_batch(Zd, lam, sigma)
        o["hv"] = nlp.eval_hessian_product_batch(Zd, lam, v, sigma)
        outs.append({k: _np(t) for k, t in o.items()})
    for k in ("f", "grad", "g", "jw", "jty", "hess", "hv"):
        assert np.isfinite(outs[0][k]).all(), k
        assert np.array_equal(outs[0][k], outs[1][k]), (k, np.argwhere(outs[0][k] != outs[1][k])[:4].tolist())


# ---- B. products at theta = 0

@pytest.mark.parametrize("im", [1, 2])
def test_products_at_theta_edges(im):
    """theta = 0 exactly (d/dtheta = +lb/2: theta > 0 is false) and +-1e-300 (tests/test_mp_reference_cpu.theta_edges).
    Row 0 has full directions; row j has w and v zero outside the j-th sampled knot, so J w and H v there are the
    model's blocks J_k w_k and H_k v_k, compared per knot."""
    pytest.importorskip("mpmath")
    from mp_nlp import Model, sample_knots
    p = ql.build_problem(N=61, k_trans=21, init_mode=im)
    nlp = ql.HybridNLP.from_problem(p, pattern="true", hessian=True, products=True)
    n, m = nlp.n_nlp, nlp.m_nlp
    z = theta_edges(p, 11)
    mdl = Model(p)
    knots = sample_knots(p.N, p.k_trans)
    assert any(z[20 * (k - 1) + 2] == 0.0 for k in knots)
    B = len(knots) + 1
    rng = np.random.default_rng(4)
    w, y, v = rng.standard_normal((B, n)), rng.standard_normal((B, m)), rng.standard_normal((B, n))
    lam, sigma = rng.standard_normal(m), 0.7
    for j, k in enumerate(knots, 1):
        off = np.ones(n, dtype=bool)
        off[20 * (k - 1):20 * (k - 1) + mdl.nvar(k)] = False
        w[j, off] = v[j, off] = 0.0
    Zd, lamd, sd = _cuda(np.tile(z, (B, 1))), _cuda(np.tile(lam, (B, 1))), _cuda(np.full(B, sigma))
    out = nlp.eval_products_batch(Zd, w=_cuda(w), y=_cuda(y))
    jw, jty = _np(out["jw"]), _np(out["jty"])
    hv = _np(nlp.eval_hessian_product_batch(Zd, lamd, _cuda(v), sigma=sd))
    vals = _np(nlp.eval_batch(Zd[:1], want=("jac",))["jac"])[0]
    hvals = _np(nlp.eval_hessian_batch(Zd[:1], lamd[:1], sd[:1]))[0]
    rows, cols = nlp.jacobian_structure_arrays()
    mr, mc, mv = mirrored(*nlp.hessian_structure_arrays(), hvals)
    for b in range(B):
        assert np.array_equal(jw[b], fold_rows(rows, cols, vals, w[b], m)), b
        assert np.array_equal(jty[b], fold_rows(rows, cols, vals, y[b], n, transpose=True)), b
        assert np.array_equal(hv[b], fold_rows(mr, mc, mv, v[b], n)), b
    for j, k in enumerate(knots, 1):
        r, Jk, _ = mdl.jac_knot(z, k)
        cs = slice(20 * (k - 1), 20 * (k - 1) + mdl.nvar(k))
        err = np.abs(jty[0][cs] - Jk.T @ y[0][r])
        assert np.all(err <= 1e-14 + 64 * EPS * (np.abs(Jk).T @ np.abs(y[0][r]))), ("J' y", k)
        want, tol = np.zeros(m), np.full(m, 1e-14)
        want[r], tol[r] = Jk @ w[j][cs], 1e-14 + 64 * EPS * (np.abs(Jk) @ np.abs(w[j][cs]))
        assert np.all(np.abs(jw[j] - want) <= tol), ("J w", k)
        # H v: the model's Hessian is held to the device values at 1e-12 of the block (check_hess), on top of the
        # rounding of the fold -- the tolerance of tests/test_products_cpu.py's model check
        Hk = mdl.hess_knot(z, k, sigma, lam)
        vk = v[j][cs]
        want, tol = np.zeros(n), np.full(n, 1e-14)
        want[cs] = Hk @ vk
        tol[cs] += (1e-12 + 64 * EPS) * (np.abs(Hk) @ np.abs(vk)) + 1e-12 * np.abs(Hk).max() * np.abs(vk).sum()
        assert np.all(np.abs(hv[j] - want) <= tol), ("H v", k)


# ---- C. KKT solve: sx = NULL, planted statuses, failures in a long batch

class Kkt:
    """B problems of one class: W = spd_w (diagonally dominant: M > 0 without sx), J the device's SPARSE_TRUE values
    at perturbed guesses, dc in [DC_MIN, 1], random right-hand sides."""
    DC_MIN = 1e-2

    def __init__(self, N, kt, im, B, seed):
        self.p = p = ql.build_problem(N=N, k_trans=kt, init_mode=im)
        self.nlp = nlp = ql.HybridNLP.from_problem(p, pattern="true", hessian=True)
        base = ql.initial_guess(p) if kt > 1 else np.zeros(p.n_nlp)
        self.jac = _np(nlp.eval_batch(_cuda(perturbed_batch(p, [base], B, 5e-2, seed)), want=("jac",))["jac"])
        self.w = spd_w(nlp, seed)
        self.hess = np.tile(self.w, (B, 1))
        rng = np.random.default_rng(seed)
        self.dc = rng.uniform(self.DC_MIN, 1.0, (B, nlp.m_nlp))
        self.r1, self.r2 = rng.standard_normal((B, nlp.n_nlp)), rng.standard_normal((B, nlp.m_nlp))

    def solve(self, sx=None):
        px, pl, st = self.nlp.kkt_solve_batch(*(_cuda(a) for a in (self.hess, self.jac, self.dc, self.r1, self.r2)),
                                              sx=None if sx is None else _cuda(sx))
        return _np(px), _np(pl), _np(st)


@pytest.mark.parametrize("N,kt,im", [(2, 2, 1), (61, 21, 1), (1024, 1000, 1)])
def test_kkt_without_sx_is_zero_sx(N, kt, im):
    B = 3
    cs = Kkt(N, kt, im, B, seed=N)
    nlp = cs.nlp
    px, pl, st = cs.solve()
    zx, zl, zs = cs.solve(sx=np.zeros((B, nlp.n_nlp)))
    assert (st == 0).all() and np.array_equal(st, zs)
    assert np.array_equal(px, zx) and np.array_equal(pl, zl)
    hs, js = nlp.hessian_structure_arrays(), nlp.jacobian_structure_arrays()
    for b in range(B):
        K = kkt_ref.kkt_matrix(hs, cs.hess[b], js, cs.jac[b], np.zeros(nlp.n_nlp), cs.dc[b])
        res, scale = kkt_ref.residual(K, px[b], pl[b], cs.r1[b], cs.r2[b])
        assert res <= 1e-12 * scale, (b, res, scale)


def _k0s(N, kt):
    return sorted({k for k in (1, 2, kt - 1, kt, 32, 33, N - 1, N) if 1 <= k <= N})


@pytest.mark.parametrize("N,kt,im", [(2, 2, 1), (61, 21, 1), (1024, 1000, 1)])
def test_planted_status_names_the_knot(N, kt, im):
    """Row j: W with a negative diagonal planted at knot k0_j (tests/test_second_order_cpu.py proves the reference's
    status is k0 for this construction); the last row is left clean."""
    k0s = _k0s(N, kt)
    B = len(k0s) + 1
    cs = Kkt(N, kt, im, B, seed=N + 1)
    for j, k0 in enumerate(k0s):
        cs.hess[j, planted_entry(cs.nlp, k0)[1]] = planted_value(cs.nlp, cs.jac[j], k0, cs.DC_MIN)
    px, pl, st = cs.solve()
    assert st.tolist() == k0s + [0]
    assert np.isnan(px[:-1]).all() and np.isnan(pl[:-1]).all()
    assert np.isfinite(px[-1]).all() and np.isfinite(pl[-1]).all()


def _dyn_entry(nlp, k0, last):
    """Index into the SPARSE_TRUE values of an entry of A_k0 (the RK4 block of step k0: a defect row of step k0, a
    column of knot k0): the first or the last of them."""
    rows, cols = nlp.jacobian_structure_arrays()
    knot = (cols - 1) // 20 + 1
    dyn = np.intersect1d(rows[knot == k0], rows[knot == k0 + 1])
    e = np.nonzero((knot == k0) & np.isin(rows, dyn))[0]
    return int(e[-1] if last else e[0])


def _w_entry(nlp, k0, last):
    """Index into the W values of an entry of knot k0's block, off the diagonal where the block has one."""
    hr, hc = nlp.hessian_structure_arrays()
    e = np.nonzero((hc - 1) // 20 + 1 == k0)[0]
    off = e[hr[e] != hc[e]]
    e = off if off.size else e
    return int(e[-1] if last else e[0])


def test_failures_in_a_long_batch_stay_local():
    """B = 16,384 at N = 61: more than 9 problems per resident warp (about 12 warps per SM x 148 SMs), so warps pick up
    a clean problem after a failed one with the shared-memory state the failure left.  Every fifth problem fails in one
    of the ways the status reports; every clean problem must have the bits it has in a batch of clean problems only,
    where it sits at another position."""
    N, kt, im, B = 61, 21, 1, 16384
    cs = Kkt(N, kt, im, 1, seed=3)
    nlp = cs.nlp
    n, m = nlp.n_nlp, nlp.m_nlp
    k0s = _k0s(N, kt)
    kinds = [("plant", k0) for k0 in k0s] + [("w-nan", k0) for k0 in k0s] + [("w-inf", k0) for k0 in k0s] + \
            [("j-nan", k0) for k0 in k0s if k0 < N] + [("j-inf", k0) for k0 in k0s if k0 < N] + \
            [("dc-inf", 0), ("dc-zero", 0), ("r1-nan", 0), ("r2-nan", 0)]
    gen = torch.Generator(device="cuda").manual_seed(7)
    hess, jac = _cuda(cs.w).repeat(B, 1), _cuda(cs.jac[0]).repeat(B, 1)
    dc = cs.DC_MIN + (1.0 - cs.DC_MIN) * torch.rand((B, m), generator=gen, dtype=F64, device="cuda")
    r1 = torch.randn((B, n), generator=gen, dtype=F64, device="cuda")
    r2 = torch.randn((B, m), generator=gen, dtype=F64, device="cuda")
    bad = np.arange(2, B, 5)
    want = np.zeros(B, dtype=np.int32)
    edits = {"hess": ([], [], []), "jac": ([], [], []), "dc": ([], [], []), "r1": ([], [], []), "r2": ([], [], [])}
    nan, inf = float("nan"), float("inf")
    for j, b in enumerate(bad.tolist()):
        kind, k0 = kinds[j % len(kinds)]
        if kind == "plant":
            t, i, x = "hess", planted_entry(nlp, k0)[1], planted_value(nlp, cs.jac[0], k0, cs.DC_MIN)
        elif kind.startswith("w-"):
            t, i, x = "hess", _w_entry(nlp, k0, kind == "w-inf"), nan if kind == "w-nan" else inf
        elif kind.startswith("j-"):
            t, i, x = "jac", _dyn_entry(nlp, k0, kind == "j-inf"), nan if kind == "j-nan" else inf
        elif kind.startswith("dc-"):
            t, i, x, k0 = "dc", (37 * j) % m, inf if kind == "dc-inf" else 0.0, -1
        else:
            t, i, x, k0 = kind[:2], (37 * j) % (n if kind == "r1-nan" else m), nan, 0
        want[b] = k0
        for lst, val in zip(edits[t], (b, i, x)):
            lst.append(val)
    arrays = {"hess": hess, "jac": jac, "dc": dc, "r1": r1, "r2": r2}
    for t, (rb, ri, rx) in edits.items():
        arrays[t][torch.tensor(rb, device="cuda"), torch.tensor(ri, device="cuda")] = torch.tensor(rx, dtype=F64, device="cuda")
    px, pl, st = nlp.kkt_solve_batch(hess, jac, dc, r1, r2)
    st_h = _np(st)
    assert np.array_equal(st_h, want), np.argwhere(st_h != want)[:8].tolist()
    failed = torch.from_numpy(np.nonzero(want != 0)[0]).cuda()
    assert bool(torch.isnan(px[failed]).all()) and bool(torch.isnan(pl[failed]).all())
    rnan = torch.from_numpy(bad[[kinds[j % len(kinds)][0] in ("r1-nan", "r2-nan") for j in range(len(bad))]]).cuda()
    assert rnan.numel() and not bool(torch.isfinite(px[rnan]).all(dim=1).any())
    clean = np.setdiff1d(np.arange(B), bad)
    perm = torch.from_numpy(np.roll(clean, 1000)).cuda()          # each clean problem at another position
    qx, ql_, qs = nlp.kkt_solve_batch(hess[perm], jac[perm], dc[perm], r1[perm], r2[perm])
    assert not bool(qs.any()) and bool(torch.isfinite(qx).all())
    assert _same_bits(px[perm], qx) and _same_bits(pl[perm], ql_)


# ---- D. poisoned rows of the Hessian and product launches

def test_poisoned_rows_stay_local_in_long_batches():
    """B = 16,384 at N = 61, NaN or Inf in one entry of Z, lambda, sigma, v, w or y of every fifth row: the Hessian, H v,
    J w, J' y and the fused f / grad / g of the clean rows are the bits of a batch of the clean rows alone."""
    p = ql.default_problem()
    nlp = ql.HybridNLP.from_problem(p, pattern="true", hessian=True, products=True)
    n, m, N, B = p.n_nlp, p.m_nlp, p.N, 16384
    gen = torch.Generator(device="cuda").manual_seed(9)
    Z = _cuda(ql.initial_guess(p)).repeat(B, 1) + 1e-2 * torch.randn((B, n), generator=gen, dtype=F64, device="cuda")
    Z[:, 19::20].clamp_(1e-3, 2e-2)
    ins = {"Z": Z, "lam": torch.randn((B, m), generator=gen, dtype=F64, device="cuda"),
           "sigma": 0.3 + 1.4 * torch.rand((B, 1), generator=gen, dtype=F64, device="cuda"),
           "v": torch.randn((B, n), generator=gen, dtype=F64, device="cuda"),
           "w": torch.randn((B, n), generator=gen, dtype=F64, device="cuda"),
           "y": torch.randn((B, m), generator=gen, dtype=F64, device="cuda")}
    # outputs a poisoned input reaches whichever entry it is (a lambda of a linear row reaches none)
    hits = {"Z": ("f",), "lam": (), "sigma": ("hess",), "v": ("hv",), "w": ("jw",), "y": ("jty",)}
    width = {"Z": n, "lam": m, "sigma": 1, "v": n, "w": n, "y": m}
    bad = np.arange(1, B, 5)
    kinds = [(t, x) for t in ins for x in (float("nan"), float("inf"))]
    for j, b in enumerate(bad.tolist()):
        t, x = kinds[j % len(kinds)]
        ins[t][b, (20 * ((7 * j) % N) + j % 20) % width[t] if t != "sigma" else 0] = x

    def run(s):
        Zs, lam, sig = ins["Z"][s], ins["lam"][s], ins["sigma"][s].reshape(-1).contiguous()
        o = nlp.eval_products_batch(Zs, w=ins["w"][s], y=ins["y"][s], want=("f", "grad", "g"))
        o["hess"] = nlp.eval_hessian_batch(Zs, lam, sig)
        o["hv"] = nlp.eval_hessian_product_batch(Zs, lam, ins["v"][s], sig)
        return o

    got = run(slice(None))
    clean = torch.from_numpy(np.setdiff1d(np.arange(B), bad)).cuda()
    alone = run(clean)
    for k, t in alone.items():
        assert bool(torch.isfinite(t).all()), k
        assert _same_bits(got[k][clean], t), k
    for j, b in enumerate(bad[:len(kinds)].tolist()):            # the poison reaches the outputs it feeds
        t, _ = kinds[j]
        for k in hits[t]:
            assert not bool(torch.isfinite(got[k][b]).all()), (t, k)
