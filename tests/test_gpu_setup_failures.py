"""Out-of-memory at every allocation a handle makes on first use.

qlnlp_debug_fail_alloc(i) makes the i-th device or pinned allocation of a handle from now on fail as an out-of-memory
cudaMalloc would.  For each first-use path, i runs over 0, 1, 2, ... until the call no longer reaches the injected
failure; each i runs once.  At every i the call must raise QLNLP_ENOMEM, the same call once disarmed must give the bits
of a handle that never saw a failure, and destroying the handles must give back every block they owned
(qlnlp_debug_owned_blocks).
"""
import ctypes as C
import itertools

import numpy as np
import pytest

import quadruped_landing_b200 as ql
from conftest import perturbed_batch
from quadruped_landing_b200 import evaluator as qev

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

B = 64


class Inputs:
    """Seeded inputs of the default problem: B decision vectors (host and device), and the operands of a KKT solve from
    a SPARSE_TRUE handle that is destroyed before any sweep starts."""

    def __init__(self):
        p = self.p = ql.default_problem()
        n, m = p.n_nlp, p.m_nlp
        rng = np.random.default_rng(17)
        self.Z = perturbed_batch(p, [ql.initial_guess(p)], B, 1e-2, 17)
        self.Zd = torch.from_numpy(self.Z).cuda()
        cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
        ref = ql.HybridNLP.from_problem(p, pattern="true", hessian=True)
        self.kkt = dict(jac=ref.eval_batch(self.Zd, want=("jac",))["jac"],
                        hess=ref.eval_hessian_batch(self.Zd, cuda(1e-4 * rng.standard_normal((B, m))),
                                                    sigma=cuda(np.full(B, 1e-4))),
                        dc=cuda(rng.uniform(1e-2, 1.0, (B, m))), r1=cuda(rng.standard_normal((B, n))),
                        r2=cuda(rng.standard_normal((B, m))), sx=cuda(rng.uniform(1.0, 10.0, (B, n))))
        _destroy(ref)
        self.rag_index = torch.arange(B, dtype=torch.int64, device="cuda")
        self.class_of = (self.rag_index >= B // 2).to(torch.int32)     # the first half in class 0, the second in class 1


@pytest.fixture(scope="module")
def inputs():
    return Inputs()


@pytest.fixture(autouse=True)
def _disarmed():
    yield
    qev.load_library().qlnlp_debug_fail_alloc(-1)


def _destroy(*nlps):
    torch.cuda.synchronize()
    for nlp in nlps:
        qev.load_library().qlnlp_destroy(nlp._h)
        nlp._h = C.c_void_p()


def _host(o):
    if isinstance(o, dict):
        return {k: _host(v) for k, v in o.items()}
    if isinstance(o, (tuple, list)):
        return tuple(_host(v) for v in o)
    if isinstance(o, torch.Tensor):
        torch.cuda.synchronize()
        return o.cpu().numpy()
    return np.array(o, copy=True)


def _assert_same_bits(got, want, what):
    if isinstance(want, dict):
        assert got.keys() == want.keys(), what
        for k in want:
            _assert_same_bits(got[k], want[k], f"{what}: {k}")
    elif isinstance(want, tuple):
        for i, (a, b) in enumerate(zip(got, want)):
            _assert_same_bits(a, b, f"{what}: [{i}]")
    else:
        assert got.dtype == want.dtype and got.shape == want.shape, what
        assert np.ascontiguousarray(got).tobytes() == np.ascontiguousarray(want).tobytes(), what


# ---- the first-use paths: make(inputs) -> fresh handles, first(inputs, handles) -> the results of their first use ----
def _single(x, nlp):
    f, grad, g, vec = np.empty(1), np.empty(nlp.n_nlp), np.empty(nlp.m_nlp), np.empty(nlp.nnz)
    nlp.eval_all(x, f, grad, g, vec)
    return f, grad, g, vec


def _dense(x, nlp):
    vec = np.empty(nlp.nnz)
    nlp.eval_constraint_jacobian(vec, x)
    return vec


def _host_batch_4_lanes(inp):
    nlp = ql.HybridNLP.from_problem(inp.p)
    nlp.set_option("host_chunk", B // 4)
    return [nlp]


def _ragged(inp, hs):
    n, m, nnz = hs[0].n_nlp, hs[0].m_nlp, hs[0].nnz
    off = {"z_off": inp.rag_index * n, "g_off": inp.rag_index * m, "j_off": inp.rag_index * nnz}
    flat = {"Z": inp.Zd.reshape(-1), "f": torch.full((B,), float("nan"), dtype=torch.float64, device="cuda"),
            "g": torch.full((B * m,), float("nan"), dtype=torch.float64, device="cuda"),
            "jac": torch.full((B * nnz,), float("nan"), dtype=torch.float64, device="cuda")}
    ql.HybridNLP.eval_ragged_classes(hs, inp.rag_index, inp.class_of, flat, off)
    return {k: flat[k] for k in ("f", "g", "jac")}


PATHS = {
    "eval_batch": (lambda inp: [ql.HybridNLP.from_problem(inp.p)], lambda inp, hs: hs[0].eval_batch(inp.Zd)),
    "eval_batch_host": (_host_batch_4_lanes, lambda inp, hs: hs[0].eval_batch_host(inp.Z)),
    "single_evaluation": (lambda inp: [ql.HybridNLP.from_problem(inp.p)], lambda inp, hs: _single(inp.Z[0], hs[0])),
    "dense_jacobian": (lambda inp: [ql.HybridNLP.from_problem(inp.p, use_sparse_jacobian=False)],
                       lambda inp, hs: _dense(inp.Z[1], hs[0])),
    "kinematic_eval_batch": (lambda inp: [ql.HybridNLP.from_problem(inp.p, kinematics=True)],
                             lambda inp, hs: hs[0].eval_batch(inp.Zd)),
    "kkt_solve_batch": (lambda inp: [ql.HybridNLP.from_problem(inp.p, pattern="true", hessian=True)],
                        lambda inp, hs: hs[0].kkt_solve_batch(**inp.kkt)),
    "ragged_classes": (lambda inp: [ql.HybridNLP.from_problem(inp.p), ql.HybridNLP.from_problem(inp.p)], _ragged),
}


@pytest.mark.parametrize("path", list(PATHS))
def test_out_of_memory_at_every_first_use_allocation(inputs, path):
    make, first = PATHS[path]
    L = qev.load_library()
    assert L.qlnlp_debug_fail_alloc(-1) == -1
    before = L.qlnlp_debug_owned_blocks()
    hs = make(inputs)
    want = _host(first(inputs, hs))
    _destroy(*hs)
    assert L.qlnlp_debug_owned_blocks() == before
    for i in itertools.count():
        hs = make(inputs)
        L.qlnlp_debug_fail_alloc(i)
        try:
            got = first(inputs, hs)
        except ql.QlnlpError as e:
            assert L.qlnlp_debug_fail_alloc(-1) == -1, f"allocation {i}: failed without reaching the injected failure"
            assert e.code == qev.QLNLP_ENOMEM, (i, str(e))
            _assert_same_bits(_host(first(inputs, hs)), want, f"{path}, retried after allocation {i} failed")
            _destroy(*hs)
            assert L.qlnlp_debug_owned_blocks() == before, f"{path}: blocks left after allocation {i} failed"
            continue
        assert L.qlnlp_debug_fail_alloc(-1) >= 0, f"allocation {i}: the injected failure was swallowed"
        _assert_same_bits(_host(got), want, path)
        _destroy(*hs)
        assert L.qlnlp_debug_owned_blocks() == before
        break
    print(f"{path}: {i} allocation points")
    assert i > 0
