"""Accuracy of the batched KKT step on the GPU at interior-point scalings, against an extended-precision solve of the full
KKT matrix (tests/kkt_hp.py): the one-shot step's backward error, the refined step (kkt_solve_refined_batch) per block,
the status at tiny dc, the residual kernel (qlnlp_kkt_residual_batch_device) entry by entry against a long-double
residual, and the refinement chain on streams and in CUDA graphs.

Regime grid (seeded): dc on the equality rows in {1e-2, 1e-6, 1e-8, 1e-10, 1e-12}; dc on the inequality rows 10^U(-2,0)
or, for an "active set", 10^U(-10,2); sx U(1,10) or 10^U(-8,8).  W and J come from the device kernels at perturbed
guesses (test_gpu_kkt.Case: sigma = multiplier scale = 1e-4).  Errors are relative to the largest entry of each block
(px, pl)."""
import time

import numpy as np
import pytest

import kkt_hp
import kkt_ref
from test_gpu_kkt import Case, _cuda, _np, _placed
from test_second_order_cpu import planted_entry, planted_w

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

EPS = kkt_hp.EPS
DC_EQ = (1e-2, 1e-6, 1e-8, 1e-10, 1e-12)
REGIMES = [(d, act, wide) for d in DC_EQ for act in (False, True) for wide in (False, True)]
CLASSES = [(2, 2, 1), (5, 3, 1), (33, 1, 2), (61, 21, 1), (61, 21, 2), (1024, 1000, 1)]
PER_CELL = 3


def _regimes(N):
    if N > 100:                                   # two problems each, three regimes: benign, tiny dc, tiny dc + wide
        return [(1e-2, False, False), (1e-12, False, False), (1e-12, True, True)], 2
    return REGIMES, PER_CELL


def _name(reg):
    d, act, wide = reg
    return f"dc_eq {d:.0e} {'active' if act else 'mild  '} sx {'wide' if wide else 'mild'}"


def _grid_case(N, kt, im, seed, **kw):
    """One batch per class: PER_CELL problems per regime, dc and sx drawn per problem (kw: Case's Z, sigma)."""
    regs, per = _regimes(N)
    B = len(regs) * per
    cs = Case(N, kt, im, B, seed=seed, **kw)
    rng = np.random.default_rng(seed + 1)
    lb, ub = cs.nlp.constraint_bounds()
    eq = lb == ub
    n, m = cs.nlp.n_nlp, cs.nlp.m_nlp
    cells = []
    for i, (d, act, wide) in enumerate(regs):
        rows = list(range(i * per, (i + 1) * per))
        for b in rows:
            ineq = 10.0 ** (rng.uniform(-10, 2, m) if act else rng.uniform(-2, 0, m))
            cs.dc[b] = np.where(eq, d, ineq)
            cs.sx[b] = 10.0 ** rng.uniform(-8, 8, n) if wide else rng.uniform(1.0, 10.0, n)
        cells.append(((d, act, wide), rows))
    return cs, cells


def _refined(cs, steps, sx=True, **kw):
    px, pl, st = cs.nlp.kkt_solve_refined_batch(cs.hess, cs.jac, _cuda(cs.dc), _cuda(cs.r1), _cuda(cs.r2),
                                                sx=_cuda(cs.sx) if sx else None, steps=steps, **kw)
    return _np(px), _np(pl), _np(st)


def _same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


# Refined step (3 steps) per regime, where it does not reach 1e-12 per block and omega <= 1e-14 at every class: the
# largest error measured over all classes on a B200 (1,000 W), times 10.  In these cells refinement against the
# condensed factor contracts by only 1e-1 .. 1e-3 a step (the factor is far from K), so three steps stop short.  At
# N <= 61 each such problem first gets the issue's allowance, 10 x Skeel's condition of K times eps; the table applies
# only beyond it, and the test prints both.  dc_eq 1e-12 with an active set and wide sx does not converge at all: there
# only "no worse than the one-shot step" is asserted (None).
STALL = {
    (1e-10, True, True): (1e-11, 5e-11),
    (1e-10, False, True): (1e-12, 5e-12),
    (1e-12, True, False): (1e-12, 2e-11),         # omega 2.3e-12 at the recorded solutions, sigma = 1
    (1e-12, False, False): (5e-10, 5e-10),        # omega 3.8e-11 at the recorded solutions, sigma = 1
    (1e-12, False, True): (1e-4, 5e-4),
    (1e-12, True, True): None,
}


def _skeel_eps(K, z):
    """|| |K^-1| |K| |z| ||_inf / ||z||_inf x eps: the forward error a backward stable solve of K can be held to
    (dense inverse; the horizons up to 61)."""
    Kd = K.toarray()
    z = np.abs(np.asarray(z, dtype=np.float64))
    return float((np.abs(np.linalg.inv(Kd)) @ (np.abs(Kd) @ z)).max() / z.max()) * EPS


def _check_grid(cs, cells, label):
    """The one-shot step and the refined step (2 and 3 steps) of every problem of the grid against kkt_solve_hp.
    One-shot: normwise backward error <= 1e-12 where dc_eq >= 1e-6 and the inequality dc are mild, <= 5e-10 elsewhere
    (measured on a B200: up to 7e-11 with an active set, 5e-12 at N = 5 with dc_eq <= 1e-8).  Refined: 1e-12 per block
    and componentwise backward error <= 1e-14, or the cell's STALL bound; and in every cell no worse than the one-shot
    step, per block (up to 1e-14) and in componentwise backward error.  Problems with a non-zero status are NaN and returned for the caller's status check."""
    N = cs.nlp.N
    n = cs.nlp.n_nlp
    px0, pl0, st0 = cs.solve()
    px2, pl2, _ = _refined(cs, 2)
    px3, pl3, st3 = _refined(cs, 3)
    assert np.array_equal(st0, st3)
    checked, failed, bad = 0, [], []

    def check(ok, *what):
        if not ok:
            bad.append((label, _name(reg)) + what)

    for reg, rows in cells:
        one, two, ref, notes = [], [], [], []
        for b in rows:
            if st0[b] != 0:
                assert np.isnan(px3[b]).all() and np.isnan(pl3[b]).all(), (b, st0[b])
                failed.append(b)
                continue
            K = cs.K(b)
            r = np.concatenate([cs.r1[b], cs.r2[b]])
            zt = kkt_hp.kkt_solve_hp(K, r, n)
            z0 = np.concatenate([px0[b], pl0[b]])
            bwd = kkt_hp.normwise_bwd(K, z0, r)
            check(bwd <= (1e-12 if reg[0] >= 1e-6 and not reg[1] else 5e-10), b, "one-shot bwd", bwd)
            e0 = kkt_hp.block_errors(z0, zt, n)
            one.append(e0 + (bwd,))
            z2 = np.concatenate([px2[b], pl2[b]])
            two.append(kkt_hp.block_errors(z2, zt, n) + (kkt_hp.componentwise_bwd(K, z2, r),))
            z3 = np.concatenate([px3[b], pl3[b]])
            ex, el = kkt_hp.block_errors(z3, zt, n)
            omega = kkt_hp.componentwise_bwd(K, z3, r)
            ref.append((ex, el, omega))
            check(ex <= max(e0[0], 1e-14) and el <= max(e0[1], 1e-14), b, "worse than one-shot", e0, ex, el)
            omega0 = kkt_hp.componentwise_bwd(K, z0, r)
            check(omega <= 1.01 * max(omega0, 1e-15), b, "omega above one-shot", omega0, omega)   # the guard's promise
            tol, otol = 1e-12, 1e-14
            if max(ex, el) > tol and N <= 61:
                sk = _skeel_eps(K, zt)
                tol = max(tol, 10.0 * sk)
                notes.append(f"b={b} Skeel x eps {sk:.1e}")
            if (max(ex, el) > tol or omega > otol) and reg in STALL:
                if STALL[reg] is None:                 # no convergence: only "no worse than one-shot" above
                    notes.append(f"b={b} not converging: px {ex:.1e}")
                    checked += 1
                    continue
                tol, otol = max(tol, STALL[reg][0]), STALL[reg][1]
                notes.append(f"b={b} stall, measured bound {tol:.0e} / {otol:.0e}")
            check(ex <= tol and el <= tol, b, "refined", ex, el, tol)
            check(omega <= otol, b, "omega", omega, otol)
            checked += 1
        if one:
            e1, e2, r3 = np.array(one), np.array(two), np.array(ref)
            print(f"{label} {_name(reg)}: one-shot px {e1[:, 0].max():.1e} pl {e1[:, 1].max():.1e} bwd {e1[:, 2].max():.1e}"
                  f" | 2 steps px {e2[:, 0].max():.1e} pl {e2[:, 1].max():.1e} omega {e2[:, 2].max():.1e}"
                  f" | 3 steps px {r3[:, 0].max():.1e} pl {r3[:, 1].max():.1e} omega {r3[:, 2].max():.1e}"
                  + (f" | status {[int(st0[b]) for b in rows if st0[b]]}" if len(one) < len(rows) else "")
                  + (" | " + "; ".join(notes) if notes else ""))
        else:
            print(f"{label} {_name(reg)}: every problem has a non-zero status {[int(st0[b]) for b in rows]}")
    assert not bad, "\n".join(map(str, bad))
    return checked, failed, st0


@pytest.mark.parametrize("N,kt,im", CLASSES)
def test_step_accuracy_against_an_extended_precision_solve(N, kt, im):
    """_check_grid over the regime grid of one class, W at sigma = multiplier scale = 1e-4 (|W| <= 0.12): every problem
    at dc_eq >= 1e-8 factors, and every checked problem meets its bound."""
    kkt_hp.require_long_double()
    t0 = time.time()
    cs, cells = _grid_case(N, kt, im, seed=100 + N + kt + im)
    checked, failed, st0 = _check_grid(cs, cells, f"N={N} kt={kt} im={im}")
    print(f"N={N} kt={kt} im={im}: {checked} problems checked, {time.time() - t0:.1f} s")
    assert checked and all(st0[b] == 0 for reg, rows in cells if reg[0] >= 1e-8 for b in rows)


def test_step_accuracy_at_the_recorded_solutions(golden):
    """The regime grid at the six recorded solutions (N = 61), sigma = 1: W is the Lagrangian Hessian at a solution,
    with the objective's x-h entries (up to ~1e3), not a small perturbation of diag(sx).  Problems that factor are held
    to _check_grid's bounds; the status of the others is the inertia of the dense M wherever its deciding leading
    block is clear of zero by 1e-9 ||M|| (as in test_gpu_kkt.py::test_status_is_the_inertia_test)."""
    kkt_hp.require_long_double()
    t0 = time.time()
    Z = np.stack([golden[f"data_{i}"] for i in range(1, 7)])
    B = len(REGIMES) * PER_CELL
    cs, cells = _grid_case(61, 21, 1, seed=500, Z=Z[np.arange(B) % 6], sigma=np.ones(B))
    checked, failed, st0 = _check_grid(cs, cells, "recorded solutions, sigma = 1")
    n, decided = cs.nlp.n_nlp, 0
    for b in failed:
        M = kkt_ref.schur_dense(cs.K(b), n)
        want = kkt_ref.status_of(M, 61)
        k = want if want else 61
        lead = M[:20 * k - (5 if k == 61 else 0), :20 * k - (5 if k == 61 else 0)]
        if abs(np.linalg.eigvalsh(lead).min()) < 1e-9 * np.abs(M).max():
            continue
        assert st0[b] == want, (b, st0[b], want)
        decided += 1
    print(f"recorded solutions: {checked} problems checked, {len(failed)} with a non-zero status ({decided} of them "
          f"decided by the dense inertia), {time.time() - t0:.1f} s")
    assert checked > 0


def _plant(cs, b, w, jv, k0):
    """W values of problem b with the negative diagonal entry of tests/test_second_order_cpu.py planted at knot k0,
    lowered by that variable's sx as well (the construction there takes sx = 0)."""
    i, e = planted_entry(cs.nlp, k0)
    w = planted_w(cs.nlp, w, jv, k0, float(cs.dc[b].min()))
    w[e] -= cs.sx[b][i]
    return w


@pytest.mark.parametrize("N,kt,im", [(5, 3, 1), (9, 4, 2)])
def test_status_is_the_inertia_test_at_interior_point_scalings(N, kt, im):
    """Every regime of the grid, with a negative W diagonal entry planted at a random knot in every other problem
    (_plant: M's entry there is below -sum J^2 / dc_min - 1 whatever sx holds): the status is the first
    knot whose leading block of the dense M is not positive definite, asserted where that block's smallest eigenvalue
    is clear of zero by 1e-9 ||M||, as in test_gpu_kkt.py::test_status_is_the_inertia_test."""
    cs, cells = _grid_case(N, kt, im, seed=7 * N)
    rng = np.random.default_rng(N)
    hess, jac = _np(cs.hess), _np(cs.jac)
    planted = {}
    for b in range(1, hess.shape[0], 2):
        planted[b] = int(rng.integers(1, N + 1))
        hess[b] = _plant(cs, b, hess[b], jac[b], planted[b])
    cs.hess = _cuda(hess)
    px, pl, st = cs.solve()
    n = cs.nlp.n_nlp
    sides, tiny_dc = set(), 0
    for reg, rows in cells:
        for b in rows:
            M = kkt_ref.schur_dense(cs.K(b), n)
            want = kkt_ref.status_of(M, N)
            k = want if want else N
            lead = M[:20 * k - (5 if k == N else 0), :20 * k - (5 if k == N else 0)]
            if abs(np.linalg.eigvalsh(lead).min()) < 1e-9 * np.abs(M).max():
                continue
            assert st[b] == want, (_name(reg), b, planted.get(b), st[b], want)
            if b in planted:
                assert 1 <= want <= planted[b]
            assert np.isnan(px[b]).all() == (want != 0) and np.isnan(pl[b]).all() == (want != 0)
            sides.add(want == 0)
            tiny_dc += reg[0] <= 1e-8
    assert sides == {True, False}
    assert tiny_dc > 0


# ---- the residual kernel

def _term_counts(nlp, with_sx):
    """Terms of each residual entry's fold, r included: s1_i = 1 + W entries of row i (mirrored) + sx + J entries of
    column i; s2_r = 1 + J entries of row r + dc."""
    n, m = nlp.n_nlp, nlp.m_nlp
    hr, hc = nlp.hessian_structure_arrays()
    jr, jc = nlp.jacobian_structure_arrays()
    t1 = np.ones(n, dtype=np.int64) + (1 if with_sx else 0)
    np.add.at(t1, hr - 1, 1)
    np.add.at(t1, (hc - 1)[hr != hc], 1)
    np.add.at(t1, jc - 1, 1)
    t2 = np.full(m, 2, dtype=np.int64)
    np.add.at(t2, jr - 1, 1)
    return t1, t2


def _residual(cs, px, pl, sx=True, **kw):
    s1, s2 = cs.nlp.kkt_residual_batch(cs.hess, cs.jac, _cuda(cs.dc), _cuda(px), _cuda(pl), _cuda(cs.r1), _cuda(cs.r2),
                                       sx=_cuda(cs.sx) if sx else None, **kw)
    return _np(s1), _np(s2)


@pytest.mark.parametrize("N,kt,im", [(2, 2, 1), (2, 1, 2), (5, 3, 1), (33, 1, 2), (61, 21, 1), (1024, 1000, 2)])
def test_residual_is_within_the_summation_bound(N, kt, im):
    """Each entry within gamma_t (|r| + |K| |z|) of the long-double residual, t its own term count, at the one-shot
    step (a residual that cancels) and at random px, pl; with and without sx, over the regime grid."""
    kkt_hp.require_long_double()
    cs, cells = _grid_case(N, kt, im, seed=300 + N + kt)
    n, m = cs.nlp.n_nlp, cs.nlp.m_nlp
    B = cs.dc.shape[0]
    rng = np.random.default_rng(N)
    px0, pl0, st0 = cs.solve()
    ok = st0 == 0
    step_px = np.where(ok[:, None], px0, rng.standard_normal((B, n)))
    step_pl = np.where(ok[:, None], pl0, rng.standard_normal((B, m)))
    rand_px = rng.standard_normal((B, n)) * 10.0 ** rng.uniform(-3, 3, (B, 1))
    rand_pl = rng.standard_normal((B, m)) * 10.0 ** rng.uniform(-3, 3, (B, 1))
    for with_sx in (True, False):
        t1, t2 = _term_counts(cs.nlp, with_sx)
        assert t1.max() <= 56 and t2.max() <= 23
        t = np.concatenate([t1, t2]).astype(np.longdouble)
        gamma = t * EPS / (1 - t * EPS)
        for what, px, pl in (("step", step_px, step_pl), ("random", rand_px, rand_pl)):
            s1, s2 = _residual(cs, px, pl, sx=with_sx)
            worst = 0.0
            for b in range(B):
                K = cs.K(b, sx=None if with_sx else np.zeros(n))
                z, r = np.concatenate([px[b], pl[b]]), np.concatenate([cs.r1[b], cs.r2[b]])
                want = kkt_hp.residual_hp(K, z, r)
                err = np.abs(np.concatenate([s1[b], s2[b]]).astype(np.longdouble) - want)
                bound = gamma * kkt_hp.abs_scale_hp(K, z, r)
                assert (err <= bound).all(), (what, with_sx, b, int(np.argmax(err - bound)))
                worst = max(worst, float((err / np.where(bound > 0, bound, 1)).max()))
            print(f"N={N} {what} sx={with_sx}: largest error / bound {worst:.2f}")


def test_residual_bits_depend_on_the_problem_alone():
    cs = Case(61, 21, 1, 1, seed=11)
    nlp = cs.nlp
    n, m = nlp.n_nlp, nlp.m_nlp
    lb, ub = nlp.constraint_bounds()
    cs.dc[0] = np.where(lb == ub, 1e-10, cs.dc[0])
    px, pl, st = cs.solve()
    assert st[0] == 0
    one = dict(hess=_np(cs.hess)[0], jac=_np(cs.jac)[0], dc=cs.dc[0], px=px[0], pl=pl[0], r1=cs.r1[0], r2=cs.r2[0],
               sx=cs.sx[0])
    ref = _residual(cs, px, pl)
    for B, pos, ld_extra, off in ((1, 0, 0, 0), (7, 3, 1, 0), (64, 63, 2, 1), (300, 150, 3, 1), (5000, 4097, 0, 1)):
        args = {k: _placed(v, B, pos, v.shape[-1] + ld_extra, off) for k, v in one.items()}
        for k in ("hess", "jac"):
            args[k][:] = args[k][pos]
        s1 = torch.full((B, n + ld_extra + off), 7.0, dtype=torch.float64, device="cuda")[:, off:off + n]
        s2 = torch.full((B, m + ld_extra + off), 7.0, dtype=torch.float64, device="cuda")[:, off:off + m]
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            nlp.kkt_residual_batch(**args, out=(s1, s2))
        side.synchronize()
        for got, want in ((_np(s1)[pos], ref[0][0]), (_np(s2)[pos], ref[1][0])):
            assert np.array_equal(got.view(np.int64), want.view(np.int64)), (B, pos)


def test_residual_writes_only_its_rows():
    cs = Case(33, 21, 2, 5, seed=2)
    n, m = cs.nlp.n_nlp, cs.nlp.m_nlp
    px, pl, _ = cs.solve()
    canary = 12345.678
    bufs = {name: torch.full((7, w + 3), canary, dtype=torch.float64, device="cuda") for name, w in (("s1", n), ("s2", m))}
    _residual(cs, px, pl, out=(bufs["s1"][1:6, 1:1 + n], bufs["s2"][1:6, 1:1 + m]))
    for name, w in (("s1", n), ("s2", m)):
        a = _np(bufs[name])
        assert (a[0] == canary).all() and (a[6] == canary).all(), name
        assert (a[1:6, 0] == canary).all() and (a[1:6, 1 + w:] == canary).all(), name
        assert np.isfinite(a[1:6, 1:1 + w]).all() and not (a[1:6, 1:1 + w] == canary).any(), name


def test_residual_of_nan_rows_is_nan_there_only():
    """A failed solve writes NaN px and pl; their residual rows are NaN, every other row is finite."""
    cs = Case(61, 21, 2, 6, seed=5)
    px, pl, st = cs.solve()
    assert (st == 0).all()
    px[[1, 4]] = np.nan
    pl[[1, 4]] = np.nan
    s1, s2 = _residual(cs, px, pl)
    for s in (s1, s2):
        assert np.isnan(s[[1, 4]]).all()
        assert np.isfinite(s[[0, 2, 3, 5]]).all()


# ---- the refinement chain

def test_refinement_chain_on_streams_and_in_graphs():
    """factor -> solve -> 3 x (residual -> factored solve -> add) on a side stream with no host synchronisation, the
    same chain captured in a CUDA graph and replayed twice: the same bits.  Rows with a non-zero factor status (a dc
    entry <= 0, a planted indefinite W) stay NaN with that status; steps = 0 gives the one-shot bits."""
    B = 16
    cs = Case(61, 21, 1, B, seed=17)
    lb, ub = cs.nlp.constraint_bounds()
    cs.dc[:] = np.where(lb == ub, 1e-8, cs.dc)
    cs.dc[3, 5] = -1.0
    hess = _np(cs.hess)
    hess[9] = _plant(cs, 9, hess[9], _np(cs.jac)[9], 4)
    cs.hess = _cuda(hess)
    one = cs.solve()
    assert one[2][3] == -1 and one[2][9] != 0
    bad = one[2] != 0
    args = dict(hess=cs.hess, jac=cs.jac, dc=_cuda(cs.dc), r1=_cuda(cs.r1), r2=_cuda(cs.r2), sx=_cuda(cs.sx))
    nlp = cs.nlp
    # steps = 0: the one-shot bits
    got = tuple(_np(t) for t in nlp.kkt_solve_refined_batch(**args, steps=0))
    for a, b in zip(got, one):
        assert _same_bits(a, b)
    # eager, default stream
    want = [t.clone() for t in nlp.kkt_solve_refined_batch(**args, steps=3)]
    torch.cuda.synchronize()
    wp, wl, ws = (_np(t) for t in want)
    assert np.array_equal(ws, one[2])
    assert np.isnan(wp[bad]).all() and np.isnan(wl[bad]).all()
    assert np.isfinite(wp[~bad]).all() and np.isfinite(wl[~bad]).all()
    assert not np.array_equal(wp[~bad], one[0][~bad])          # refinement changed the step
    # a side stream, no host synchronisation in between
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        got = nlp.kkt_solve_refined_batch(**args, steps=3)
    side.synchronize()
    for a, b in zip(got, want):
        assert _same_bits(_np(a), _np(b))
    # captured (after the eager calls above warmed the handle), replayed twice
    outs = [torch.empty_like(t) for t in want]
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        nlp.kkt_solve_refined_batch(**args, steps=3, out=tuple(outs))
    for rep in range(2):
        for o in outs:
            o.fill_(float("nan")) if o.dtype == torch.float64 else o.fill_(-9)
        torch.cuda.synchronize()
        g.replay()
        torch.cuda.synchronize()
        for a, b in zip(outs, want):
            assert _same_bits(_np(a), _np(b)), rep
