"""The CUDA outputs held to the extended-precision model of the NLP (tests/mp_nlp.py) through every entry point, with
the helpers and tolerances the CPU tests hold the oracle to, and the long horizons up to N = 1024 (32 passes of one lane
per knot): bit identity with the oracle on every row, the model on sampled knots (every pass boundary, the jump, the
end), canary rows around padded outputs, host batches over several pipeline chunks, the Hessian and ragged launches."""
import numpy as np
import pytest

from conftest import perturbed_batch
from oracle.oracle import Oracle
import quadruped_landing_b200 as ql

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
pytest.importorskip("mpmath")
from mp_nlp import Model, check_f, check_g, check_grad, check_hess, check_jac, check_jac_dense, sample_knots  # noqa: E402
from test_gpu_parity import assert_same_bits  # noqa: E402
from test_mp_reference_cpu import hess_knots, random_point, random_problem, theta_edges  # noqa: E402

_models = {}


def model(prob, key, **kw):
    """One model per problem and boundary states: its per-knot results are reused by every entry point."""
    if key not in _models:
        _models[key] = Model(prob, **kw)
    return _models[key]


def check_row(m, z, out, rows, cols, knots, b=0):
    """f, grad, g and the Jacobian of row ``b`` of a batch's outputs against the model."""
    check_f(m, z, out["f"][b])
    check_grad(m, z, out["grad"][b])
    check_g(m, z, out["g"][b], knots)
    check_jac(m, z, out["jac"][b], rows, cols, knots)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(out):
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items() if isinstance(v, torch.Tensor)}


@pytest.fixture(scope="module")
def rnd():
    """The problem with nothing at its default, per-evaluation boundary states, and a batch whose rows 0 and 1 the
    model checks."""
    p = random_problem(17)
    rng = np.random.default_rng(3)
    B = 70
    Z = np.stack([random_point(p, 100 + b) for b in range(B)])
    x0, xf = rng.normal(size=(B, 15)), rng.normal(size=(B, 15))
    x0[1], xf[1] = p.x0, p.xf
    return p, Z, x0, xf


def rnd_model(p, x0, xf, b):
    return model(p, ("rnd", b), x0=x0[b], xf=xf[b])


@pytest.mark.parametrize("ieee_div", [False, True])
@pytest.mark.parametrize("pattern", ["block", "true"])
def test_eval_batch(rnd, pattern, ieee_div, monkeypatch):
    """Both patterns, both division instantiations, per-evaluation x0 / xf, the random problem."""
    if ieee_div:
        monkeypatch.setenv("QLNLP_IEEE_DIV", "1")
    p, Z, x0, xf = rnd
    nlp, o = ql.HybridNLP.from_problem(p, pattern=pattern), Oracle(p)
    out = host(nlp.eval_batch(dev(Z), x0=dev(x0), xf=dev(xf)))
    assert_same_bits(nlp, out, o.eval_batch(Z, x0=x0, xf=xf, pattern=pattern))
    rows, cols = nlp.jacobian_structure_arrays()
    for b in (0, 1):
        check_row(rnd_model(p, x0, xf, b), Z[b], out, rows, cols, sample_knots(p.N, p.k_trans), b)


def test_default_problem_at_theta_edges():
    """theta = 0 and +-1e-300 (Q4) at the default instance, both patterns."""
    p = ql.default_problem()
    z = theta_edges(p, 7)
    m = model(p, "theta")
    for pattern in ("block", "true"):
        nlp = ql.HybridNLP.from_problem(p, pattern=pattern)
        out = host(nlp.eval_batch(dev(np.stack([z, z]))))
        check_row(m, z, out, *nlp.jacobian_structure_arrays(), range(1, p.N + 1), 1)


def test_single_evaluation_entry_points(rnd):
    """The four MOI callbacks, eval_all, and the DENSE grid with its zeros."""
    p, Z, _, _ = rnd
    z, m = Z[1], model(p, ("rnd", 1), x0=p.x0, xf=p.xf)
    knots = range(1, p.N + 1)
    for pattern in ("block", "true"):
        nlp = ql.HybridNLP.from_problem(p, pattern=pattern)
        rows, cols = nlp.jacobian_structure_arrays()
        check_f(m, z, nlp.eval_objective(z))
        grad, g, vals = np.empty(nlp.n_nlp), np.empty(nlp.m_nlp), np.empty(nlp.nnz)
        nlp.eval_objective_gradient(grad, z)
        nlp.eval_constraint(g, z)
        nlp.eval_constraint_jacobian(vals, z)
        check_row(m, z, {"f": [nlp.eval_objective(z)], "grad": [grad], "g": [g], "jac": [vals]}, rows, cols, knots)
        f, grad, g, vals = np.empty(1), np.empty(nlp.n_nlp), np.empty(nlp.m_nlp), np.empty(nlp.nnz)
        nlp.set_option("x_cache", 0)
        nlp.eval_all(z, f, grad, g, vals)
        check_row(m, z, {"f": f, "grad": [grad], "g": [g], "jac": [vals]}, rows, cols, knots)
    dn = ql.HybridNLP.from_problem(p, use_sparse_jacobian=False)
    vec = np.full(dn.nnz, np.nan)
    dn.eval_constraint_jacobian(vec, z)
    check_jac_dense(m, z, vec.reshape(dn.n_nlp, dn.m_nlp).T, knots)


def test_host_batch_compact_transfer(rnd):
    """eval_batch_host with B >= 64: only the value-dependent Jacobian entries cross PCIe, host threads rebuild rows."""
    p, Z, x0, xf = rnd
    for pattern in ("block", "true"):
        nlp = ql.HybridNLP.from_problem(p, pattern=pattern)
        out = nlp.eval_batch_host(Z, x0=x0, xf=xf)
        assert_same_bits(nlp, out, Oracle(p).eval_batch(Z, x0=x0, xf=xf, pattern=pattern))
        rows, cols = nlp.jacobian_structure_arrays()
        for b in (0, 1):
            check_row(rnd_model(p, x0, xf, b), Z[b], out, rows, cols, sample_knots(p.N, p.k_trans), b)


def test_kinematic_handle():
    p = ql.build_problem(N=33, k_trans=12, init_mode=2)
    Z = perturbed_batch(p, [ql.initial_guess(p)], 8, 5e-2, 4)
    m = model(p, "kin", kinematics=True)
    for pattern in ("block", "true"):
        nlp = ql.HybridNLP.from_problem(p, pattern=pattern, kinematics=True)
        out = host(nlp.eval_batch(dev(Z)))
        rows, cols = nlp.jacobian_structure_arrays()
        check_g(m, Z[0], out["g"][0])
        check_jac(m, Z[0], out["jac"][0], rows, cols, range(1, p.N + 1))


def _ragged(probs, vecs, x0, xf):
    """One qlnlp_eval_ragged_classes launch with per-problem x0 / xf; returns the rows of every problem."""
    ev = ql.RaggedEvaluator(probs)
    class_of = np.arange(len(probs))
    plan = ev.plan(class_of)
    Zd = dev(ev.pack(class_of, vecs))
    off = plan.off
    flat = {"Z": Zd, "f": torch.empty(len(probs), dtype=torch.float64, device="cuda")}
    for k, o in (("grad", "z_off"), ("g", "g_off"), ("jac", "j_off")):
        flat[k] = torch.full((int(off[o][-1]),), np.nan, dtype=torch.float64, device="cuda")
    ql.HybridNLP.eval_ragged_classes(ev.nlps, plan.order, plan.dclass, flat, plan.doff, x0=dev(x0), xf=dev(xf),
                                     z_padded=True)
    out = host(flat)
    res = []
    for i, e in enumerate(ev.nlps):
        sl = lambda k, o, w: out[k][off[o][i]:off[o][i] + w][None, :]
        res.append((e, {"f": out["f"][i:i + 1], "grad": sl("grad", "z_off", e.n_nlp), "g": sl("g", "g_off", e.m_nlp),
                        "jac": sl("jac", "j_off", e.nnz_block)}))
    return res


def test_ragged_classes_with_their_own_tables_and_states():
    """Classes with random model constants and cost tables, per-problem x0 / xf, the largest horizon not first."""
    probs = [random_problem(40 + i, N, kt, im) for i, (N, kt, im) in enumerate([(9, 4, 2), (61, 21, 1), (2, 1, 1), (33, 33, 2)])]
    rng = np.random.default_rng(8)
    vecs = [random_point(p, 50 + i) for i, p in enumerate(probs)]
    x0, xf = rng.normal(size=(len(probs), 15)), rng.normal(size=(len(probs), 15))
    for i, (e, got) in enumerate(_ragged(probs, vecs, x0, xf)):
        p = probs[i]
        assert_same_bits(e, got, Oracle(p).eval_batch(vecs[i][None, :], x0=x0[i:i + 1], xf=xf[i:i + 1]))
        check_row(model(p, ("ragged", i), x0=x0[i], xf=xf[i]), vecs[i], got, *e.jacobian_structure_arrays(),
                  sample_knots(p.N, p.k_trans))


def test_hessian_batch(rnd, monkeypatch):
    """sigma given and default (1); an output with odd leading dimension (plain stores) and an even one, both with
    guard rows; lambda rows wider than m_nlp; and the single host-pointer call.  Both division instantiations: one
    handle created without QLNLP_IEEE_DIV and one with it (the variable is read once, when a handle is created)."""
    p, Z, _, _ = rnd
    nlps = []
    for ieee_div in (False, True):
        monkeypatch.delenv("QLNLP_IEEE_DIV", raising=False)
        if ieee_div:
            monkeypatch.setenv("QLNLP_IEEE_DIV", "1")
        nlps.append(ql.HybridNLP.from_problem(p, hessian=True))
    monkeypatch.delenv("QLNLP_IEEE_DIV", raising=False)
    B, guard, sentinel = 6, 2, -7.25
    rng = np.random.default_rng(9)
    lam_wide = dev(rng.standard_normal((B, p.m_nlp + 3)))
    lam = lam_wide[:, :p.m_nlp]                                  # ldlambda = m_nlp + 3
    sigma = rng.uniform(0.3, 1.7, size=B)
    knots = hess_knots(p.N, p.k_trans) + [5, 17]
    m = model(p, ("rnd", 1), x0=p.x0, xf=p.xf)
    for nlp in nlps:
        rows, cols = nlp.hessian_structure_arrays()
        nh = nlp.nnz_hess
        for sig in (sigma, None):
            for pad in (nh % 2 + 1, 2 - nh % 2):                 # odd and even leading dimension
                big = torch.full((B + 2 * guard, nh + pad), sentinel, dtype=torch.float64, device="cuda")
                H = nlp.eval_hessian_batch(dev(Z[:B]), lam, None if sig is None else dev(sig),
                                           out=big[guard:guard + B, :nh])
                torch.cuda.synchronize()
                assert bool((big[:guard] == sentinel).all()) and bool((big[guard + B:] == sentinel).all())
                assert bool((big[:, nh:] == sentinel).all()) and not bool((H == sentinel).any())
                s = 1.0 if sig is None else sig[1]
                check_hess(m, Z[1], s, lam[1].cpu().numpy(), H[1].cpu().numpy(), rows, cols, knots)
        vals = np.empty(nh)
        nlp.eval_hessian_lagrangian(vals, Z[1], sigma[1], lam[1].cpu().numpy())
        check_hess(m, Z[1], sigma[1], lam[1].cpu().numpy(), vals, rows, cols, knots)


LARGE = [(128, 33, 1), (129, 129, 2), (257, 100, 1), (1024, 2, 2), (1024, 1000, 1)]


@pytest.mark.parametrize("pattern", ["block", "true"])
@pytest.mark.parametrize("N,kt,im", LARGE)
def test_large_horizons(N, kt, im, pattern):
    p = ql.build_problem(N=N, k_trans=kt, init_mode=im)
    nlp, o = ql.HybridNLP.from_problem(p, pattern=pattern), Oracle(p)
    knots = sample_knots(N, kt)
    base = ql.initial_guess(p) if kt > 1 else np.zeros(p.n_nlp)
    B = 72
    Z = perturbed_batch(p, [base], B, 5e-2, N + kt)
    m = model(p, ("large", N, kt, im))
    ref = o.eval_batch(Z, pattern=pattern)
    rows, cols = nlp.jacobian_structure_arrays()
    # device batch: padded leading dimensions, canary rows
    guard, sentinel = 2, -7.25
    widths = {"grad": nlp.n_nlp, "g": nlp.m_nlp, "jac": nlp.nnz_batch}
    big = {k: torch.full((B + 2 * guard, w + 3), sentinel, dtype=torch.float64, device="cuda") for k, w in widths.items()}
    views = {k: big[k][guard:guard + B, :w] for k, w in widths.items()}
    views["f"] = torch.empty(B, dtype=torch.float64, device="cuda")
    got = host(nlp.eval_batch(dev(Z), out=views))
    for k, w in widths.items():
        assert bool((big[k][:guard] == sentinel).all()) and bool((big[k][guard + B:] == sentinel).all()), k
        assert bool((big[k][:, w:] == sentinel).all()), k
    del big, views
    assert_same_bits(nlp, got, ref)
    check_row(m, Z[0], got, rows, cols, knots)
    # host batch over three pipeline chunks (B >= 64: compact transfer)
    nlp.set_option("host_chunk", 32)
    hb = nlp.eval_batch_host(Z)
    for k in ("f", "grad", "g", "jac"):
        assert np.array_equal(hb[k], got[k]), k
    del hb, got, ref
    if pattern == "true":
        return
    # the Hessian at the jump, the ends and one pass boundary
    hn = ql.HybridNLP.from_problem(p, hessian=True)
    hr, hc = hn.hessian_structure_arrays()
    lam = np.random.default_rng(N).standard_normal((2, p.m_nlp))
    H = hn.eval_hessian_batch(dev(Z[:2]), dev(lam), dev(np.array([0.5, 1.5]))).cpu().numpy()
    check_hess(m, Z[0], 0.5, lam[0], H[0], hr, hc, sorted(set(hess_knots(N, kt)) | {32, 33}))
    # a ragged launch mixing the long class with short ones
    probs = [ql.build_problem(N=5, k_trans=3, init_mode=1), p, ql.build_problem(N=2, k_trans=1, init_mode=2)]
    vecs = [perturbed_batch(probs[0], [ql.initial_guess(probs[0])], 1, 1e-2, 1)[0], Z[0], np.zeros(probs[2].n_nlp)]
    x0 = np.stack([q.x0 for q in probs])
    xf = np.stack([q.xf for q in probs])
    for i, (e, r) in enumerate(_ragged(probs, vecs, x0, xf)):
        assert_same_bits(e, r, Oracle(probs[i]).eval_batch(vecs[i][None, :]))
    if N == 257:
        # the DENSE grid (N = 1024 would be 2.9 GB)
        dn = ql.HybridNLP.from_problem(p, use_sparse_jacobian=False)
        vec = np.full(dn.nnz, np.nan)
        dn.eval_constraint_jacobian(vec, Z[0])
        check_jac_dense(m, Z[0], vec.reshape(dn.n_nlp, dn.m_nlp).T, knots)
