"""Ragged launches (qlnlp_eval_ragged_classes, qlnlp_eval_ragged_device) at every layout the C ABI accepts, held bit for
bit to the strided evaluator on every row.

The reference for a problem is ``eval_batch`` of its class's handle on the same vector and boundary states.  Ragged
and strided launches run the same kernel text in the same operation order, so every row of f, grad, g and jac must
have the same bits.  One row per class is also held to the oracle; rows of the random-constants class and of the
N = 1,024 class to the extended-precision model.  After every launch every output double outside the evaluated rows
(gaps, the tail, rows and f entries of problems not in ``index``) must still hold the sentinel.

Layouts (``flat_layout`` in tests/test_ragged_cpu.py):
  padded  even row starts and QLNLP_RAGGED_Z_PADDED: TMA loads and stores on every row (the control);
  packed  rows back to back: aligned and unaligned jac rows meet in one warp, so bulk and plain stores alternate;
          Z unpadded (8-byte cp.async staging);
  gapped  1 to 3 doubles between rows and every array 8 bytes past a 16-byte boundary: plain stores only, no waits.

The five classes differ in everything a class swap replaces: (61, 21, 1) at default costs, (2, 1, 2), a problem with
its own model constants, cost tables and default x0 / xf (third, so a launch reading hs[0]'s record for it fails),
(33, 33, 1), and (65, 2, 2) across a pass boundary.  Cases of ``test_mixed_classes``, each for both patterns:

  case        entry    layout  want          order                 x0 / xf    problems (evaluated)
  control     classes  padded  all four      by class (plan order) per row    3,000
  shuffled    classes  packed  all four      random permutation    defaults   3,000
  null_index  classes  gapped  g, jac        index = NULL          per row    600
  subset      classes  packed  f, grad, g    odd problems only     per row    3,000 (1,500)
  jac_only    classes  gapped  jac           random permutation    defaults   600
  g_only      classes  packed  g             by class (plan order) per row    600
  tiny        classes  gapped  all four      random permutation    per row    3 (fewer than the classes)
  device      device   packed  all four      index = NULL          per row    300, one class
  device_sub  device   gapped  f, grad, g    odd problems reversed defaults   300 (150), one class

``f, grad, g`` without the Jacobian is the JM_NONE kernel with the late ticket.  ``test_longest_class_not_first``
mixes N = 1,024 with N = 2 (the shared-memory layout comes from the largest class, which is not hs[0]);
``test_ieee_division_fallback`` runs a table that falls back to the IEEE-division kernel because one class has it.
"""
import ctypes as C

import numpy as np
import pytest

from conftest import perturbed_batch
from oracle.oracle import Oracle
import quadruped_landing_b200 as ql
from quadruped_landing_b200 import evaluator as qev

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
pytest.importorskip("mpmath")
from mp_nlp import sample_knots  # noqa: E402
from test_gpu_mp_reference import check_row, model  # noqa: E402
from test_gpu_parity import assert_same_bits  # noqa: E402
from test_mp_reference_cpu import random_problem  # noqa: E402
from test_ragged_cpu import SENTINEL, covered, flat_layout  # noqa: E402

ALL = ("f", "grad", "g", "jac")
TABLE = {"grad": "z", "g": "g", "jac": "jac"}       # the offset table that addresses each output
Z_PADDED = 1                                          # QLNLP_RAGGED_Z_PADDED
_oracles = {}


def oracle(p):
    if id(p) not in _oracles:
        _oracles[id(p)] = (p, Oracle(p))
    return _oracles[id(p)][1]


@pytest.fixture(scope="module")
def five():
    probs = [ql.build_problem(N=61, k_trans=21, init_mode=1), ql.build_problem(N=2, k_trans=1, init_mode=2),
             random_problem(23), ql.build_problem(N=33, k_trans=33, init_mode=1),
             ql.build_problem(N=65, k_trans=2, init_mode=2)]
    ev = ql.RaggedEvaluator(probs)            # SPARSE_BLOCK handles; its plan() gives the launch order by class
    return ev, {"block": ev.nlps, "true": [ql.HybridNLP.from_problem(p, pattern="true") for p in probs]}


def guarded(n, misaligned):
    """n doubles inside a larger allocation filled with the sentinel: (the whole allocation as int64, the doubles);
    ``misaligned``: the doubles start 8 bytes past a 16-byte boundary."""
    big = torch.full((n + 2,), SENTINEL, dtype=torch.int64, device="cuda")
    assert big.data_ptr() % 16 == 0
    s = int(misaligned)
    return big, big[s:s + n].view(torch.float64)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def run(nlps, class_of, want, kind, order, x0xf, seed, entry="classes", subset=False, ev=None, model_classes=()):
    """Lay the problems out in ``kind``, launch once, and check every evaluated row against its class's strided
    evaluation (bit equality), one row per class against the oracle, the rows of ``model_classes`` against the
    model, and the sentinel everywhere else."""
    class_of = np.asarray(class_of, dtype=np.int64)
    nprob, rng, mis = class_of.size, np.random.default_rng(seed), kind == "gapped"
    Z = [None] * nprob
    for c, e in enumerate(nlps):
        ids = np.nonzero(class_of == c)[0]
        if ids.size == 0:
            continue
        p = e.prob
        base = ql.initial_guess(p) if p.k_trans > 1 else np.zeros(p.n_nlp)
        for i, z in zip(ids, perturbed_batch(p, [base], ids.size, 5e-2, seed + c)):
            Z[i] = z
    width = lambda a: np.array([getattr(nlps[c], a) for c in class_of], dtype=np.int64)
    widths = {"z": width("n_nlp"), "g": width("m_nlp"), "jac": width("nnz_batch")}
    off = {k: flat_layout(w, kind, seed + j) for j, (k, w) in enumerate(widths.items())}
    _, Zd = guarded(int(off["z"][-1]), mis)
    zhost = np.full(int(off["z"][-1]), SENTINEL, dtype=np.int64).view(np.float64)     # Z's gaps hold NaNs too
    for i, z in enumerate(Z):
        zhost[off["z"][i]:off["z"][i] + z.size] = z
    Zd.copy_(dev(zhost))

    rows = np.arange(1, nprob, 2) if subset else np.arange(nprob)
    if order == "plan":
        plan = ev.plan(class_of).order.cpu().numpy()
        index = plan[np.isin(plan, rows)]
    elif order == "random":
        index = rng.permutation(rows)
    elif order == "reversed":
        index = rows[::-1].copy()
    else:
        assert order == "null" and not subset
        index = None
    evaluated = rows if index is None else index
    if kind == "packed" and "jac" in want and len(nlps) > 1 and evaluated.size > 50:   # bulk and plain rows mix
        assert set(off["jac"][evaluated] % 2) == {0, 1}

    guards, out = {}, {}
    for k in want:
        n = nprob if k == "f" else int(off[TABLE[k]][-1])
        guards[k], out[k] = guarded(n, mis)
    x0 = xf = None
    if x0xf:
        x0, xf = rng.normal(size=(nprob, 15)), rng.normal(size=(nprob, 15))
    keep = {k: dev(v) for k, v in off.items()}               # alive until the launch has completed
    io = qev._BatchIO()
    io.Z = Zd.data_ptr()
    for k, t in out.items():
        setattr(io, k, t.data_ptr())
    if x0xf:
        keep["x0"], keep["xf"] = dev(x0), dev(xf)
        io.x0, io.xf = keep["x0"].data_ptr(), keep["xf"].data_ptr()
    if index is not None:
        keep["index"] = dev(index.astype(np.int64))
    rg = qev._RaggedIO(keep["index"].data_ptr() if index is not None else None, keep["z"].data_ptr(),
                       keep["g"].data_ptr() if "g" in want else None, keep["jac"].data_ptr() if "jac" in want else None,
                       Z_PADDED if kind == "padded" else 0)
    B = evaluated.size
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    L = ql.load_library()
    if entry == "classes":
        hs = (C.c_void_p * len(nlps))(*[e._h.value for e in nlps])
        keep["cls"] = dev(class_of.astype(np.int32))
        qev._check(L.qlnlp_eval_ragged_classes(hs, len(nlps), B, C.byref(io), C.byref(rg),
                                               C.c_void_p(keep["cls"].data_ptr()), stream))
    else:
        assert len(nlps) == 1
        qev._check(L.qlnlp_eval_ragged_device(nlps[0]._h, B, C.byref(io), C.byref(rg), stream))
    torch.cuda.synchronize()

    # canaries: nothing outside the evaluated rows was written
    for k, big in guards.items():
        if k == "f":
            inside = np.zeros(nprob, dtype=bool)
            inside[evaluated] = True
        else:
            inside = covered(off[TABLE[k]], widths[TABLE[k]], evaluated)
        full = np.zeros(big.numel(), dtype=bool)
        full[int(mis):int(mis) + inside.size] = inside
        rest = big[dev(~full)]
        assert bool((rest == SENTINEL).all()), f"{k}: {int((rest != SENTINEL).sum())} doubles written outside the rows"

    for c, e in enumerate(nlps):
        pis = np.sort(evaluated[class_of[evaluated] == c])
        if pis.size == 0:
            continue
        what = f"class {c} (N={e.N}, {e.pattern}): "
        kw = {} if x0 is None else {"x0": dev(x0[pis]), "xf": dev(xf[pis])}
        ref = e.eval_batch(dev(np.stack([Z[i] for i in pis])), want=want, **kw)
        for k in ("grad", "g", "jac"):
            if k in want:
                w = ref[k].shape[1]
                at = dev(off[TABLE[k]][pis])[:, None] + torch.arange(w, device="cuda")
                same = out[k][at].view(torch.int64) == ref[k].view(torch.int64)
                assert bool(same.all()), f"{what}{k}: rows of problems {pis[~same.all(1).cpu().numpy()][:8]} differ"
        if "f" in want:
            same = out["f"][dev(pis)].view(torch.int64) == ref["f"].view(torch.int64)
            assert bool(same.all()), f"{what}f of problems {pis[~same.cpu().numpy()][:8]} differs"
        # the first row of the class against the oracle (and the model)
        i = int(pis[0])
        got = {"f": out["f"][i:i + 1].cpu().numpy()} if "f" in want else {}
        for k in ("grad", "g", "jac"):
            if k in want:
                o = int(off[TABLE[k]][i])
                got[k] = out[k][o:o + int(widths[TABLE[k]][i])].cpu().numpy()[None, :]
        bx = {} if x0 is None else {"x0": x0[i:i + 1], "xf": xf[i:i + 1]}
        assert_same_bits(e, got, oracle(e.prob).eval_batch(Z[i][None, :], want=want, pattern=e.pattern, **bx), what)
        if c in model_classes:
            assert set(want) == set(ALL)
            m = model(e.prob, ("ragged", e.N, e.k_trans, e.init_mode, seed, i), **({} if x0 is None else {"x0": x0[i], "xf": xf[i]}))
            check_row(m, Z[i], got, *e.jacobian_structure_arrays(), sample_knots(e.N, e.k_trans))


def mixed(nprob, ncls, seed):
    """Class of each problem, every class present when there is room for it."""
    rng = np.random.default_rng(seed)
    class_of = rng.integers(0, ncls, size=nprob)
    class_of[:min(nprob, ncls)] = rng.permutation(ncls)[:min(nprob, ncls)]
    return rng.permutation(class_of)


CASES = {   # name: (entry, layout, want, order, x0 / xf per row, problems, subset)
    "control": ("classes", "padded", ALL, "plan", True, 3000, False),
    "shuffled": ("classes", "packed", ALL, "random", False, 3000, False),
    "null_index": ("classes", "gapped", ("g", "jac"), "null", True, 600, False),
    "subset": ("classes", "packed", ("f", "grad", "g"), "plan", True, 3000, True),
    "jac_only": ("classes", "gapped", ("jac",), "random", False, 600, False),
    "g_only": ("classes", "packed", ("g",), "plan", True, 600, False),
    "tiny": ("classes", "gapped", ALL, "random", True, 3, False),
    "device": ("device", "packed", ALL, "null", True, 300, False),
    "device_sub": ("device", "gapped", ("f", "grad", "g"), "reversed", False, 300, True),
}


@pytest.mark.parametrize("pattern", ["block", "true"])
@pytest.mark.parametrize("case", list(CASES))
def test_mixed_classes(five, case, pattern):
    ev, nlps = five
    entry, kind, want, order, x0xf, nprob, subset = CASES[case]
    seed = 1000 + list(CASES).index(case)
    if entry == "device":            # one handle: the random-constants class alone
        run([nlps[pattern][2]], np.zeros(nprob, dtype=np.int64), want, kind, order, x0xf, seed, entry, subset)
    else:
        run(nlps[pattern], mixed(nprob, 5, seed), want, kind, order, x0xf, seed, entry, subset, ev,
            model_classes=(2,) if case == "control" else ())


@pytest.mark.parametrize("pattern", ["block", "true"])
def test_longest_class_not_first(pattern):
    """N = 1,024 after N = 2: the launch's shared-memory layout must come from the largest class, not from hs[0]."""
    probs = [ql.build_problem(N=2, k_trans=1, init_mode=1), ql.build_problem(N=1024, k_trans=1000, init_mode=1)]
    nlps = [ql.HybridNLP.from_problem(p, pattern=pattern) for p in probs]
    class_of = np.array([0, 1, 0, 0, 1, 0, 0, 0, 1, 0, 0, 1, 0, 0, 0, 0])
    run(nlps, class_of, ALL, "packed", "random", True, 77, model_classes=(1,))


@pytest.mark.parametrize("pattern", ["block", "true"])
def test_ieee_division_fallback(five, pattern, monkeypatch):
    """One class created with QLNLP_IEEE_DIV: the whole launch runs the IEEE-division kernel, and every row still
    equals its class's strided evaluation, whose handles use the reciprocal-FMA division where it is exact."""
    _, nlps = five
    monkeypatch.setenv("QLNLP_IEEE_DIV", "1")
    ieee = ql.HybridNLP.from_problem(random_problem(29), pattern=pattern)
    monkeypatch.delenv("QLNLP_IEEE_DIV")
    run(nlps[pattern][:2] + [ieee], mixed(300, 3, 5), ALL, "packed", "random", True, 88)
