"""The oracle, and the host emulation of the generated device code, held to the extended-precision model of the NLP
(tests/mp_nlp.py).  Bit-identity tests elsewhere tie the kernels to the oracle; these tie the oracle to the mathematics,
so an error the two share (a misplaced column, a sign, a wrong row at the jump knot, an entry missing from a pattern)
fails here.  The tolerances are the ones the GPU tests use (tests/test_gpu_mp_reference.py)."""
import numpy as np
import pytest

from oracle.oracle import Oracle
import quadruped_landing_b200 as ql

pytest.importorskip("mpmath")
from mp_nlp import Model, check_f, check_g, check_grad, check_hess, check_jac, check_jac_dense, sample_knots  # noqa: E402

CLASSES = [(2, 1, 1), (2, 2, 2), (3, 2, 2), (5, 3, 1), (9, 4, 2), (33, 33, 1), (33, 1, 2), (61, 21, 1), (61, 21, 2)]


def perturbed(prob, seed, sigma=5e-2):
    rng = np.random.default_rng(seed)
    base = ql.initial_guess(prob) if prob.k_trans > 1 else np.zeros(prob.n_nlp)
    z = base + sigma * rng.standard_normal(prob.n_nlp)
    z[19::20] = np.clip(z[19::20], 1e-3, 2e-2)
    return z


def theta_edges(prob, seed):
    """theta = 0 exactly at every third knot (Q4: d/dtheta = +lb/2 there), +-1e-300 at the others."""
    z = perturbed(prob, seed)
    th = z[2::20]
    th[0::3] = 0.0
    th[1::3] = 1e-300
    th[2::3] = -1e-300
    return z


def random_problem(seed, N=37, kt=12, im=2):
    """A problem with nothing at its default: model constants, per-knot cost tables (R55 != 0, so the h entries of the
    gradient are not 0), boundary states."""
    rng = np.random.default_rng(seed)
    model = ql.PlanarQuadruped(g=-3.71 - rng.random(), mb=7.3 + rng.random(), mf=0.23 + 0.1 * rng.random(),
                               lb=0.61 + 0.1 * rng.random(), l1=0.3, l2=0.2)
    obj = [ql.LQRCost(rng.uniform(0, 20, 15), rng.uniform(0, 1, 5), rng.normal(size=15), rng.normal(size=5) * 30)
           for _ in range(N)]
    return ql.ProblemData.from_costs(model, obj, im, kt, N, rng.normal(size=15), rng.normal(size=15))


def random_point(prob, seed):
    rng = np.random.default_rng(seed)
    z = rng.normal(size=prob.n_nlp)
    z[19::20] = rng.uniform(1e-3, 2e-2, size=prob.N - 1)
    return z


def hess_knots(N, kt):
    return sorted({k for k in (1, kt - 1, kt, N - 1, N) if 1 <= k <= N})


def _emul_streams(emul_lib, prob, z):
    m = prob.model
    nlp = ql.HybridNLP.from_problem(prob)
    segs = nlp._debug_segments()
    block = np.empty(nlp.nnz)
    assert emul_lib.emul_jac_stream(prob.N, prob.k_trans, prob.init_mode, m.g, m.mb, m.mf, m.lb, segs.ctypes.data,
                                    len(segs), z.ctypes.data, block.ctypes.data, 1) == 0
    nlp_t = ql.HybridNLP.from_problem(prob, pattern="true")
    true = np.empty(nlp_t.nnz)
    assert emul_lib.emul_true_stream(prob.N, prob.k_trans, prob.init_mode, m.g, m.mb, m.mf, m.lb, z.ctypes.data,
                                     true.ctypes.data, nlp_t.nnz) == 0
    return (nlp, block), (nlp_t, true)


def _check_all(emul_lib, prob, z, knots, x0=None, xf=None):
    """f, grad, g, both sparse patterns (oracle and emulated device stream) and, for short horizons, the dense grid."""
    o, mdl = Oracle(prob), Model(prob, x0=x0, xf=xf)
    bx0 = None if x0 is None else x0[None, :]
    bxf = None if xf is None else xf[None, :]
    ref = o.eval_batch(z[None, :], x0=bx0, xf=bxf)
    check_f(mdl, z, ref["f"][0])
    check_grad(mdl, z, ref["grad"][0])
    check_g(mdl, z, ref["g"][0])
    refs = {"block": ref["jac"][0], "true": o.eval_batch(z[None, :], x0=bx0, xf=bxf, pattern="true")["jac"][0]}
    for (nlp, emul), pattern in zip(_emul_streams(emul_lib, prob, z), ("block", "true")):
        rows, cols = nlp.jacobian_structure_arrays()
        check_jac(mdl, z, refs[pattern], rows, cols, knots)
        check_jac(mdl, z, emul, rows, cols, knots)
    if prob.N <= 9:
        check_jac_dense(mdl, z, o.jac_c_dense(z), knots)
    return mdl


@pytest.mark.parametrize("N,kt,im", CLASSES)
def test_oracle_and_device_streams_against_the_model(emul_lib, N, kt, im):
    prob = ql.build_problem(N=N, k_trans=kt, init_mode=im)
    knots = sample_knots(N, kt, every=33)
    _check_all(emul_lib, prob, perturbed(prob, 10 * N + kt), knots)
    z = theta_edges(prob, 10 * N + kt + 1)
    mdl = _check_all(emul_lib, prob, z, knots)
    # the Hessian: oracle (dense second-order forward mode) and the generated device code
    rng = np.random.default_rng(N + kt)
    lam, sigma = rng.standard_normal(prob.m_nlp), float(rng.uniform(0.3, 1.7))
    nlp = ql.HybridNLP.from_problem(prob, hessian=True)
    rows, cols = nlp.hessian_structure_arrays()
    hk = hess_knots(N, kt)
    check_hess(mdl, z, sigma, lam, Oracle(prob).hess_lagrangian_dense(z, sigma, lam)[rows - 1, cols - 1], rows, cols, hk)
    out = np.empty(nlp.nnz_hess)
    m = prob.model
    assert emul_lib.emul_hess_stream(N, kt, im, m.g, m.mb, m.mf, m.lb, prob.Q.ctypes.data, prob.R.ctypes.data,
                                     prob.q.ctypes.data, prob.r.ctypes.data, z.ctypes.data, sigma, lam.ctypes.data,
                                     out.ctypes.data, nlp.nnz_hess) == 0
    check_hess(mdl, z, sigma, lam, out, rows, cols, hk)


def test_recorded_solution(golden, emul_lib):
    prob = ql.default_problem()
    _check_all(emul_lib, prob, golden["data_6"].copy(), sample_knots(prob.N, prob.k_trans))


@pytest.mark.parametrize("N,kt,im", [(37, 12, 2), (9, 4, 1)])
def test_random_problem_with_its_own_boundary_states(emul_lib, N, kt, im):
    """Random model constants and per-knot cost tables, and per-evaluation x0 / xf that differ from the problem's."""
    prob = random_problem(17 + N, N, kt, im)
    z = random_point(prob, 18 + N)
    rng = np.random.default_rng(N)
    mdl = _check_all(emul_lib, prob, z, sample_knots(N, kt), x0=rng.normal(size=15), xf=rng.normal(size=15))
    lam, sigma = rng.standard_normal(prob.m_nlp), 0.8
    nlp = ql.HybridNLP.from_problem(prob, hessian=True)
    rows, cols = nlp.hessian_structure_arrays()
    check_hess(mdl, z, sigma, lam, Oracle(prob).hess_lagrangian_dense(z, sigma, lam)[rows - 1, cols - 1], rows, cols,
               hess_knots(N, kt))


@pytest.mark.parametrize("N,kt,im", [(5, 3, 1), (9, 4, 2), (33, 1, 2)])
def test_kinematic_rows(N, kt, im):
    prob = ql.build_problem(N=N, k_trans=kt, init_mode=im)
    o, mdl = Oracle(prob, kinematics=True), Model(prob, kinematics=True)
    z = perturbed(prob, N)
    ref = o.eval_batch(z[None, :])
    check_g(mdl, z, ref["g"][0])
    knots = sample_knots(N, kt)
    for pattern in ("block", "true"):
        rows, cols = ql.HybridNLP.from_problem(prob, pattern=pattern, kinematics=True).jacobian_structure_arrays()
        check_jac(mdl, z, o.eval_batch(z[None, :], pattern=pattern)["jac"][0], rows, cols, knots)


@pytest.mark.parametrize("N,kt,im", CLASSES)
def test_sparse_true_is_inside_sparse_block(N, kt, im):
    """SPARSE_TRUE is a sub-pattern of SPARSE_BLOCK; the model's non-zeros lie in SPARSE_TRUE (check_jac, above)."""
    prob = ql.build_problem(N=N, k_trans=kt, init_mode=im)
    rb, cb = ql.HybridNLP.from_problem(prob).jacobian_structure_arrays()
    rt, ct = ql.HybridNLP.from_problem(prob, pattern="true").jacobian_structure_arrays()
    m = prob.m_nlp
    assert np.isin((ct - 1) * m + rt, (cb - 1) * m + rb).all()


def test_planted_defects_are_caught():
    """The comparisons must reject small, plausible errors made on a copy of the oracle's output: this is the evidence
    that the tolerances are tight enough."""
    prob = random_problem(5, N=9, kt=4, im=2)
    o, mdl = Oracle(prob), Model(prob)
    z = random_point(prob, 6)
    N, kt = prob.N, prob.k_trans
    knots = list(range(1, N + 1))
    ref = o.eval_batch(z[None, :])
    jac, grad = ref["jac"][0], ref["grad"][0]
    rows, cols = ql.HybridNLP.from_problem(prob).jacobian_structure_arrays()
    check_jac(mdl, z, jac, rows, cols, knots)
    check_grad(mdl, z, grad)
    caught = []

    def expect_rejected(name, fn, *args):
        with pytest.raises(AssertionError):
            fn(*args)
        caught.append(name)

    # 1. one Jacobian value (an RK4-block entry of a middle knot) off by 1 part in 1e9
    k = 3
    run = np.nonzero((cols - 1) // 20 == k - 1)[0]
    i = run[np.argmax(np.abs(jac[run]) * ((rows[run] > 29) & (np.abs(jac[run]) < 1.0)))]
    bad = jac.copy()
    bad[i] *= 1 + 1e-9
    expect_rejected("value", check_jac, mdl, z, bad, rows, cols, [k])
    # 2. two adjacent, different values of one knot's run swapped
    diff = np.nonzero(np.diff(jac[run]) != 0)[0]
    j = run[diff[len(diff) // 2]]
    bad = jac.copy()
    bad[[j, j + 1]] = bad[[j + 1, j]]
    expect_rejected("swap", check_jac, mdl, z, bad, rows, cols, [k])
    # 3. the Q2 zeroing left out: the time row of the jump knot's RK4 block holds d(t + h) = 1 at t and h
    kj = kt - 1
    trow = 29 + 15 * (kj - 1) + 15
    bad = jac.copy()
    bad[(rows == trow) & ((cols == 20 * (kj - 1) + 15) | (cols == 20 * kj))] = 1.0
    expect_rejected("Q2", check_jac, mdl, z, bad, rows, cols, [kj])
    # 4. an h entry of the gradient replaced by the true derivative (Q1)
    bad = grad.copy()
    bad[20 * (k - 1) + 19] = mdl.grad_h_true(z, k)
    expect_rejected("Q1", check_grad, mdl, z, bad)
    # 5. one Hessian entry of the smallest-scale knot block off by 1 part in 1e9
    rng = np.random.default_rng(1)
    lam, sigma = rng.standard_normal(prob.m_nlp), 0.9
    nlp = ql.HybridNLP.from_problem(prob, hessian=True)
    hr, hc = nlp.hessian_structure_arrays()
    H = o.hess_lagrangian_dense(z, sigma, lam)[hr - 1, hc - 1]
    check_hess(mdl, z, sigma, lam, H, hr, hc, knots)
    scale = [np.abs(H[(hc - 1) // 20 == kk - 1]).max() for kk in knots]
    ks = knots[int(np.argmin(scale))]
    blk = np.nonzero((hc - 1) // 20 == ks - 1)[0]
    bad = H.copy()
    bad[blk[np.argmax(np.abs(H[blk]))]] *= 1 + 1e-9
    expect_rejected("hessian", check_hess, mdl, z, sigma, lam, bad, hr, hc, [ks])
    assert caught == ["value", "swap", "Q2", "Q1", "hessian"]
