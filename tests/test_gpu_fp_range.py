"""The kernels at the ends of the double range.

Rows scaled towards the subnormals (x, u and h times 2^-990 ... 2^-1018), single entries at subnormals and -0.0, forces
of 1e306 to 1.5e308, and body angles far outside one turn, mixed with ordinary rows in one batch per class.  Through
every path that divides by a model constant, the IEEE-division instantiations (QLNLP_IEEE_DIV) must give the oracle's
values wherever the oracle is finite, and the default FASTDIV ones what csrc/fastdiv.h documents against them: the
same values on ordinary and large-angle rows (sign of zero aside), the parity tolerance on rows pushed below 2^-969,
and NaN as the only other outcome where a*r overflows.  CUDA's sin / cos at large arguments (the slow argument
reduction) are held to the extended-precision model, and the extreme rows must not change the bits of the ordinary
rows."""
import os

import numpy as np
import pytest

from conftest import perturbed_batch
from oracle.oracle import Oracle
import quadruped_landing_b200 as ql

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
pytest.importorskip("mpmath")
import mp_nlp  # noqa: E402
from mp_nlp import Model, check_g, check_hess, check_jac, sample_knots  # noqa: E402
from test_gpu_mp_reference import _ragged  # noqa: E402
from test_gpu_second_order import _handle  # noqa: E402
from test_mp_reference_cpu import perturbed, random_problem  # noqa: E402

EPS = np.finfo(np.float64).eps
TINY = [2.0 ** -990, 2.0 ** -1000, 2.0 ** -1010, 2.0 ** -1018]
THETAS = [1e3, -1e3, 1e8, -1e8, 1e15, -1e15, 1e22, -1e22, 1e300, -1e300]
# (N, k_trans, init_mode): both initial modes, the shortest horizon and the longest (32 passes of one lane per knot)
CLASSES = [(61, 21, 1), (61, 21, 2), (2, 2, 1), (1024, 1000, 1)]
KINDS = ["plain", "tiny0", "tiny1", "tiny2", "tiny3", "entry", "huge", "theta"]


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _np(t):
    torch.cuda.synchronize()
    return t.cpu().numpy()


def edge_row(p, kind, seed):
    """One decision vector of ``kind``."""
    rng = np.random.default_rng(seed)
    z = perturbed(p, seed)
    z[2::20] *= np.where(rng.random(p.N) < 0.5, -1.0, 1.0)                    # both theta branches (Q4)
    if kind.startswith("tiny"):
        return z * TINY[int(kind[-1])]
    if kind == "entry":
        i = rng.choice(p.n_nlp, 8, replace=False)
        z[i] = [5e-324, -5e-324, 2.0 ** -1060, -2.0 ** -1030, 2.0 ** -1022, -0.0, -0.0, 5e-324]
    elif kind == "huge":
        for k in range(p.N - 1):
            z[20 * k + 15:20 * k + 19] = np.minimum(10.0 ** rng.uniform(306, 308.2, 4), 1.5e308) * \
                np.where(rng.random(4) < 0.5, -1.0, 1.0)
    elif kind == "theta":
        z[2::20] = rng.choice(THETAS, p.N)
    return z


def edge_batch(p, B, seed):
    return np.stack([edge_row(p, KINDS[b % len(KINDS)], seed + b) for b in range(B)])


def assert_bits(got, want, what):
    """Equal NaN masks and equal int64 views elsewhere: the sign of zero and +-Inf count."""
    got, want = np.asarray(got), np.asarray(want)
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan), (what, np.argwhere(np.isnan(got) != nan)[:4].tolist())
    bad = (got.view(np.int64) != want.view(np.int64)) & ~nan
    assert not bad.any(), (what, np.argwhere(bad)[:4].tolist(), got[bad][:4], want[bad][:4])


def assert_oracle_bits(nlp, got, ref, what=""):
    """tests/test_gpu_parity.assert_same_bits where the oracle is finite: equal values outside the sin / cos entries,
    4 ulp(1) on them (their operands are O(1)).  The oracle's dense duals overflow at huge inputs where the kernels'
    sparse code does not."""
    N = nlp.N
    for k in ("f", "grad", "g", "jac"):
        a, b = np.asarray(got[k]), np.asarray(ref[k])
        trig = np.zeros(b.shape[-1], dtype=bool)
        if k == "g":
            trig[nlp.m_nlp - N:] = True
        elif k == "jac":
            rows, cols = nlp.jacobian_structure_arrays()
            trig = (rows > nlp.m_nlp - N) & ((cols - 1) % 20 == 2)
        fin = np.isfinite(b)
        exact = fin & ~trig if k != "f" else fin
        assert np.array_equal(a[exact], b[exact]), (what, k, np.argwhere(exact & (a != b))[:4].tolist())
        if k != "f":
            t = fin & trig
            assert np.all(np.abs(a[t] - b[t]) <= 4 * EPS), (what, k)


def assert_documented(fast, ieee, kind, what):
    """One row of a FASTDIV output against the IEEE-division one, by the kind of the row (csrc/fastdiv.h)."""
    fast, ieee = np.asarray(fast, dtype=np.float64), np.asarray(ieee, dtype=np.float64)
    nan = np.isnan(ieee)
    assert np.isnan(fast[nan]).all(), (what, kind)
    if kind in ("plain", "theta"):                          # every division inside the domain
        assert np.array_equal(fast, ieee, equal_nan=True), (what, kind, np.argwhere(fast != ieee)[:4].tolist())
        return
    differ = (fast != ieee) & ~(np.isnan(fast) & nan)
    if kind == "huge":                                      # a*r overflows: NaN where IEEE gives +-Inf or a value
        assert np.isnan(fast[differ]).all(), (what, kind, fast[differ][:4], ieee[differ][:4])
    else:                                                   # numerators below 2^-969: an ulp per division
        a, b = fast[differ], ieee[differ]
        assert np.all(np.abs(a - b) <= 1e-14 + 1e-12 * np.abs(b)), (what, kind, a[:4], b[:4])


class Pair:
    """The FASTDIV and the IEEE-division handles of one problem, compared row by row."""

    def __init__(self, p, **kw):
        self.h = {ieee: _handle(p, ieee, **kw) for ieee in (False, True)}

    def compare(self, fn, what, kinds):
        """``kinds``: the kind of each row of a batch output, or one kind for a single call's output."""
        fast, ieee = (fn(self.h[i]) for i in (False, True))
        fast, ieee = (o if isinstance(o, dict) else {"": o} for o in (fast, ieee))
        for k in fast:
            if isinstance(kinds, str):
                assert_documented(fast[k], ieee[k], kinds, (what, k))
            else:
                for b, kind in enumerate(kinds):
                    assert_documented(fast[k][b], ieee[k][b], kind, (what, k, b))
        return fast, ieee


def _host(out):
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items() if isinstance(v, torch.Tensor)}


@pytest.mark.parametrize("N,kt,im", CLASSES)
def test_division_instantiations_at_the_ends_of_the_range(N, kt, im):
    """Every path that divides by a model constant: eval_batch (SPARSE_BLOCK, SPARSE_TRUE, no Jacobian), the host
    batch (VALS stream), the products (J w, J' y and the fused f / grad / g), the Hessian and H v, and the MOI single
    callbacks.  The IEEE-division outputs of eval_batch against the oracle."""
    p = ql.build_problem(N=N, k_trans=kt, init_mode=im)
    B = 64                                                  # the host batch's compact (VALS) transfer starts at 64
    Z = edge_batch(p, B, 1000 * N + im)
    kinds = [KINDS[b % len(KINDS)] for b in range(B)]
    n, m = p.n_nlp, p.m_nlp
    rng = np.random.default_rng(N)
    lam, v, w, y = (rng.standard_normal((B, d)) for d in (m, n, n, m))
    sigma = rng.uniform(0.3, 1.7, B)
    Zd, lamd, vd, wd, yd, sd = (_cuda(a) for a in (Z, lam, v, w, y, sigma))
    o = Oracle(p)
    for pattern in ("block", "true"):
        pair = Pair(p, pattern=pattern, hessian=True, products=True)
        _, ieee = pair.compare(lambda h: _host(h.eval_batch(Zd)), ("eval_batch", pattern), kinds)
        assert_oracle_bits(pair.h[True], ieee, o.eval_batch(Z, pattern=pattern), pattern)
        pair.compare(lambda h: h.eval_batch_host(Z), ("eval_batch_host", pattern), kinds)
        if pattern == "true":
            continue
        pair.compare(lambda h: _host(h.eval_batch(Zd, want=("f", "grad", "g"))), "no Jacobian", kinds)
        pair.compare(lambda h: _host(h.eval_products_batch(Zd, w=wd, y=yd, want=("f", "grad", "g"))), "products", kinds)
        pair.compare(lambda h: _np(h.eval_hessian_batch(Zd, lamd, sd)), "hessian", kinds)
        pair.compare(lambda h: _np(h.eval_hessian_product_batch(Zd, lamd, vd, sd)), "H v", kinds)
        for b in range(len(KINDS)):                          # one row of each kind through the single callbacks
            def single(h, z=Z[b]):
                out = {"f": np.array([h.eval_objective(z)]), "grad": np.empty(n), "g": np.empty(m),
                       "jac": np.empty(h.nnz), "hess": np.empty(h.nnz_hess), "jw": np.empty(m), "jty": np.empty(n),
                       "hv": np.empty(n)}
                h.eval_objective_gradient(out["grad"], z)
                h.eval_constraint(out["g"], z)
                h.eval_constraint_jacobian(out["jac"], z)
                h.eval_hessian_lagrangian(out["hess"], z, sigma[b], lam[b])
                h.eval_constraint_jacobian_product(out["jw"], z, w[b])
                h.eval_constraint_jacobian_transpose_product(out["jty"], z, y[b])
                h.eval_hessian_lagrangian_product(out["hv"], z, v[b], sigma[b], lam[b])
                return out
            pair.compare(single, "single callbacks", KINDS[b])


@pytest.mark.parametrize("kind", KINDS)
def test_ragged_launch_at_the_ends_of_the_range(kind):
    """A two-class ragged launch, one class with random model constants and cost tables, on rows of each kind."""
    probs = [ql.build_problem(N=61, k_trans=21, init_mode=1), random_problem(23, 37, 12, 2)]
    vecs = [edge_row(q, kind, 70 + i) for i, q in enumerate(probs)]
    x0, xf = np.stack([q.x0 for q in probs]), np.stack([q.xf for q in probs])
    res = []
    old = os.environ.pop("QLNLP_IEEE_DIV", None)
    try:
        for ieee in (False, True):
            if ieee:
                os.environ["QLNLP_IEEE_DIV"] = "1"
            res.append(_ragged(probs, vecs, x0, xf))
    finally:
        os.environ.pop("QLNLP_IEEE_DIV", None)
        if old is not None:
            os.environ["QLNLP_IEEE_DIV"] = old
    for i, ((_, fast), (e, ieee)) in enumerate(zip(*res)):
        for k in ("f", "grad", "g", "jac"):
            assert_documented(fast[k][0], ieee[k][0], kind, (i, k))
        assert_oracle_bits(e, ieee, Oracle(probs[i]).eval_batch(vecs[i][None, :]), (kind, i))


def test_mpmath_reduces_large_arguments():
    """The model's sin / cos at the angles below: sin(1e22) is a published value, and 60 digits agree with 720."""
    with mp_nlp.mp.workdps(mp_nlp.DPS):
        assert mp_nlp.mp.nstr(mp_nlp.mp.sin(mp_nlp.mp.mpf(1e22)), 20) == "-0.85220084976718880177"
        lo = [(mp_nlp.mp.sin(mp_nlp.mp.mpf(t)), mp_nlp.mp.cos(mp_nlp.mp.mpf(t))) for t in THETAS]
    with mp_nlp.mp.workdps(720):
        for t, (s, c) in zip(THETAS, lo):
            assert abs(mp_nlp.mp.sin(mp_nlp.mp.mpf(t)) - s) < 1e-50 and abs(mp_nlp.mp.cos(mp_nlp.mp.mpf(t)) - c) < 1e-50


@pytest.mark.parametrize("im", [1, 2])
def test_large_theta_against_the_model(im, monkeypatch):
    """theta = +-1e3 ... +-1e300 at the sampled knots: g, the Jacobian of those knots (the body row's -+lb/2 cos(theta)
    among it) and the Hessian blocks (+-lam lb/2 sin(theta) at (theta, theta), the Q4 sign) against the model.  The model runs at
    720 digits: its finite differences in theta must resolve a step of 1e-18 next to theta^2 = 1e600 in the cost."""
    monkeypatch.setattr(mp_nlp, "DPS", 720)
    p = ql.build_problem(N=61, k_trans=21, init_mode=im)
    knots = sample_knots(p.N, p.k_trans)
    z = perturbed(p, 40 + im)
    for j, k in enumerate(knots):
        z[20 * (k - 1) + 2] = THETAS[j % len(THETAS)]
    nlp = ql.HybridNLP.from_problem(p, hessian=True)
    lam = np.random.default_rng(im).standard_normal(p.m_nlp)
    out = _host(nlp.eval_batch(_cuda(z[None, :])))
    H = _np(nlp.eval_hessian_batch(_cuda(z[None, :]), _cuda(lam[None, :]), _cuda(np.array([0.7]))))[0]
    mdl = Model(p)
    check_g(mdl, z, out["g"][0], knots)
    rows, cols = nlp.jacobian_structure_arrays()
    check_jac(mdl, z, out["jac"][0], rows, cols, knots)
    hr, hc = nlp.hessian_structure_arrays()
    check_hess(mdl, z, 0.7, lam, H, hr, hc, knots)
    # check_hess scales its tolerance by the block's largest entry, which d2(h cost)/dtheta dh = 2 h Q theta makes
    # huge: hold the (theta, theta) entries to 1e-12 of themselves
    for k in knots:
        e = np.nonzero((hr == hc) & (hr == 20 * (k - 1) + 3))[0]
        want = mdl.hess_knot(z, k, 0.7, lam)[2, 2]
        assert abs(H[e[0]] - want) <= 1e-14 + 1e-12 * abs(want), (k, H[e[0]], want)


def test_extreme_rows_leave_ordinary_rows_alone():
    """B = 8,192 at N = 61 (several rows per resident warp) with every second row extreme: the ordinary rows have the bits of a batch of ordinary rows
    alone, through eval_batch, the products and the Hessian."""
    p = ql.default_problem()
    nlp = ql.HybridNLP.from_problem(p, hessian=True, products=True)
    B, n, m = 8192, p.n_nlp, p.m_nlp
    plain = perturbed_batch(p, [ql.initial_guess(p)], B // 2, 5e-2, 5)
    extreme = np.stack([edge_row(p, KINDS[1 + b % (len(KINDS) - 1)], 9000 + b) for b in range(64)])
    Z = np.empty((B, n))
    Z[0::2] = plain
    Z[1::2] = extreme[np.arange(B // 2) % 64]
    rng = np.random.default_rng(6)
    lam, v, w, y = (_cuda(rng.standard_normal((B, d))) for d in (m, n, n, m))
    sig = _cuda(rng.uniform(0.3, 1.7, B))

    def run(s):
        Zs = _cuda(Z[s])
        o = dict(nlp.eval_batch(Zs))
        o.update({"p_" + k: t for k, t in nlp.eval_products_batch(Zs, w=w[s], y=y[s], want=("f", "grad", "g")).items()})
        sg = sig[s].contiguous()
        o["hess"] = nlp.eval_hessian_batch(Zs, lam[s], sg)
        o["hv"] = nlp.eval_hessian_product_batch(Zs, lam[s], v[s], sg)
        return _host(o)

    mixed, alone = run(slice(None)), run(slice(0, None, 2))
    for k, t in alone.items():
        assert np.isfinite(t).all(), k
        assert_bits(mixed[k][0::2], t, k)
