"""One handle on several streams at once, mixed-kernel chains on one stream, and CUDA-graph replays.

The ticketed kernels (evaluator, products, Hessian, Hessian products, KKT solve) share state between launches: a work
counter pair that the last CTA of every grid re-arms, and the KKT factor and kinematic-row scratch.  Eager launches take
the counter and scratch of their stream; a launch captured into a graph takes a counter and scratch its graph owns.
Each test here makes launches meet on that state and compares every result, bit for bit, with the same launch made
alone on a quiet device.  Those one-at-a-time launches are themselves held to their references: the oracle's bits
for f / grad / g / jac, the fold of the materialised values for the products, the oracle's Hessian, and the residual
of the sparse KKT system (tests/kkt_ref.py) with status 0 for the KKT solve.  Outputs are prefilled with NaN, so a
ticket that a grid skipped shows up as unwritten rows.

Grids are kept short (B of a few hundred at N = 61) so that several of them are resident on the GPU together, and the
number of rounds is fixed: the overlap is structural, not hunted for.
"""
import ctypes as C
import os

import numpy as np
import pytest

import kkt_ref
from conftest import perturbed_batch
from oracle.oracle import Oracle
import quadruped_landing_b200 as ql
from quadruped_landing_b200 import evaluator as qev

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
from test_gpu_parity import assert_same_bits  # noqa: E402
from test_products_cpu import fold_rows, mirrored  # noqa: E402

ALL = ("f", "grad", "g", "jac")
_rigs = {}


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _nan_like(t):
    """A NaN-filled (int32: -7) tensor of t's shape with the library's row stride."""
    if t.dtype == torch.int32:
        return torch.full_like(t, -7)
    if t.dim() == 1:
        return torch.full_like(t, float("nan"))
    return torch.full((t.shape[0], t.stride(0)), float("nan"), dtype=t.dtype, device=t.device)[:, :t.shape[1]]


def _nan_tree(o):
    if isinstance(o, dict):
        return {k: _nan_tree(v) for k, v in o.items()}
    if isinstance(o, tuple):
        return tuple(_nan_tree(v) for v in o)
    return _nan_like(o)


def _clone_tree(o):
    if isinstance(o, dict):
        return {k: _clone_tree(v) for k, v in o.items()}
    if isinstance(o, tuple):
        return tuple(_clone_tree(v) for v in o)
    return o.clone()


def _fill_nan(o):
    if isinstance(o, dict):
        for v in o.values():
            _fill_nan(v)
    elif isinstance(o, tuple):
        for v in o:
            _fill_nan(v)
    else:
        o.fill_(-7 if o.dtype == torch.int32 else float("nan"))


def _assert_equal_tree(got, want, what):
    """Same bits (NaN == NaN: the references have none, so a NaN in `got` is a row left unwritten)."""
    if isinstance(want, dict):
        assert got.keys() == want.keys(), what
        for k in want:
            _assert_equal_tree(got[k], want[k], f"{what}.{k}")
    elif isinstance(want, tuple):
        for i, (a, b) in enumerate(zip(got, want)):
            _assert_equal_tree(a, b, f"{what}[{i}]")
    else:
        if not torch.equal(got, want):
            bad = (got != want) if got.dtype == torch.int32 else ~((got == want) | (got.isnan() & want.isnan()))
            rows = bad.reshape(bad.shape[0], -1).any(dim=1).nonzero().flatten()
            unwritten = got.isnan().reshape(got.shape[0], -1).all(dim=1).sum().item() if got.is_floating_point() else 0
            raise AssertionError(f"{what}: {rows.numel()} of {got.shape[0]} rows differ ({unwritten} left unwritten), "
                                 f"first {rows[:8].tolist()}")


class _RawStreams:
    """Distinct CUDA streams (torch.cuda.Stream() hands out a small pool of streams round-robin, fewer than the
    library's work-counter pool), created and destroyed through the CUDA runtime that torch has loaded."""

    def __init__(self, n):
        torch.cuda.init()
        try:
            self.rt = C.CDLL("libcudart.so.12")
        except OSError:
            import nvidia.cuda_runtime
            self.rt = C.CDLL(os.path.join(list(nvidia.cuda_runtime.__path__)[0], "lib", "libcudart.so.12"))
        self.rt.cudaStreamCreateWithFlags.argtypes = [C.POINTER(C.c_void_p), C.c_uint]
        self.rt.cudaStreamDestroy.argtypes = [C.c_void_p]
        self.raw = []
        for _ in range(n):
            s = C.c_void_p()
            assert self.rt.cudaStreamCreateWithFlags(C.byref(s), 1) == 0      # cudaStreamNonBlocking
            self.raw.append(s)
        self.streams = [torch.cuda.ExternalStream(s.value) for s in self.raw]

    def close(self):
        torch.cuda.synchronize()
        for s in self.raw:
            self.rt.cudaStreamDestroy(s)


class Rig:
    """The handles of the default problem (SPARSE_BLOCK, SPARSE_TRUE with the Hessian and products, kinematic rows),
    two seeded input sets ("parities" 0 and 1) at batch size B, and the one-at-a-time result of every launch family
    on each, held to its reference.  With ieee_div the handles run the IEEE-division kernels (QLNLP_IEEE_DIV)."""

    def __init__(self, ieee_div, B=600):
        self.ieee_div = ieee_div
        p = self.p = ql.default_problem()
        old = os.environ.pop("QLNLP_IEEE_DIV", None)
        try:
            if ieee_div:
                os.environ["QLNLP_IEEE_DIV"] = "1"
            self.blk = ql.HybridNLP.from_problem(p)
            self.tru = ql.HybridNLP.from_problem(p, pattern="true", hessian=True, products=True)
            self.kin = ql.HybridNLP.from_problem(p, kinematics=True)
        finally:
            os.environ.pop("QLNLP_IEEE_DIV", None)
            if old is not None:
                os.environ["QLNLP_IEEE_DIV"] = old
        self.B = B
        n, m = p.n_nlp, p.m_nlp
        rng = np.random.default_rng(31)
        self.Z = [perturbed_batch(p, [ql.initial_guess(p)], B, s, seed) for s, seed in ((1e-2, 5), (2e-2, 6))]
        self.Zd = [_cuda(z) for z in self.Z]
        self.lam = 1e-4 * rng.standard_normal((B, m))
        self.sigma = np.full(B, 1e-4)
        self.dc, self.sx = rng.uniform(1e-2, 1.0, (B, m)), rng.uniform(1.0, 10.0, (B, n))
        self.lamd, self.sigmad, self.dcd, self.sxd = (_cuda(a) for a in (self.lam, self.sigma, self.dc, self.sx))
        # the ragged launch: every problem of the flat batch, in reverse order, rows back to back
        self.rag_index = torch.arange(B - 1, -1, -1, dtype=torch.int64, device="cuda")
        self.rag_off = {"z_off": torch.arange(B, dtype=torch.int64, device="cuda") * n,
                        "g_off": torch.arange(B, dtype=torch.int64, device="cuda") * m,
                        "j_off": torch.arange(B, dtype=torch.int64, device="cuda") * self.blk.nnz}
        self.ref = [None, None]
        self.ref[1] = self.alone(1, jt_prev=None)        # parity 1 first: the KKT solve of parity 0 reads its jac
        self.ref[0] = self.alone(0, jt_prev=self.ref[1]["jt"]["jac"])
        self.ref[1] = self.alone(1, jt_prev=self.ref[0]["jt"]["jac"])
        for par in (0, 1):
            self.check_reference(par)

    # ---- the launches: each enqueues one library call on the current stream into `out` ----
    def new_out(self):
        B, n, m, p = self.B, self.p.n_nlp, self.p.m_nlp, self.p
        like = lambda w, dt=torch.float64: _nan_like(torch.empty((B, qev.even_ld(w)), dtype=dt, device="cuda")[:, :w])
        return {"eb": {"f": _nan_like(torch.empty(B, dtype=torch.float64, device="cuda")), "grad": like(n), "g": like(m),
                       "jac": like(self.blk.nnz)},
                "pr": {"f": _nan_like(torch.empty(B, dtype=torch.float64, device="cuda")), "g": like(m), "jw": like(m),
                       "jty": like(n)},
                "h": like(self.tru.nnz_hess), "hv": like(n),
                "kkt": (like(n), like(m), torch.full((B,), -7, dtype=torch.int32, device="cuda")),
                "jt": {"f": _nan_like(torch.empty(B, dtype=torch.float64, device="cuda")), "grad": like(n), "g": like(m),
                       "jac": like(self.tru.nnz)},
                "rag": {"f": torch.full((B,), float("nan"), dtype=torch.float64, device="cuda"),
                        "g": torch.full((B * m,), float("nan"), dtype=torch.float64, device="cuda"),
                        "jac": torch.full((B * self.blk.nnz,), float("nan"), dtype=torch.float64, device="cuda")},
                "kin": {"f": _nan_like(torch.empty(B, dtype=torch.float64, device="cuda")), "grad": like(n),
                        "g": like(self.kin.m_nlp), "jac": like(self.kin.nnz)}}

    def chain(self, par, out, jt_prev):
        """The eight launch families back to back, each reading what an earlier one wrote (the products take the
        SPARSE_BLOCK evaluation's grad and g as w and y, the Hessian product the products' J'y as v, the KKT solve the
        Hessian, the Hessian product and J w as W, r1 and r2) or overwriting what an earlier one read (the SPARSE_TRUE
        evaluation rewrites the Jacobian the KKT solve read: jt_prev is out["jt"]["jac"] in a chain)."""
        Z = self.Zd[par]
        self.blk.eval_batch(Z, out=out["eb"])
        self.tru.eval_products_batch(Z, w=out["eb"]["grad"], y=out["eb"]["g"], want=("f", "g"), out=out["pr"])
        self.tru.eval_hessian_batch(Z, self.lamd, sigma=self.sigmad, out=out["h"])
        self.tru.eval_hessian_product_batch(Z, self.lamd, out["pr"]["jty"], sigma=self.sigmad, out=out["hv"])
        self.tru.kkt_solve_batch(out["h"], jt_prev, self.dcd, out["hv"], out["pr"]["jw"], sx=self.sxd, out=out["kkt"])
        self.tru.eval_batch(Z, out=out["jt"])
        self.blk.eval_ragged(self.rag_index, {"Z": Z.view(-1), **out["rag"]}, self.rag_off)
        self.kin.eval_batch(Z, out=out["kin"])

    def alone(self, par, jt_prev):
        """Every launch of `chain` made alone: a device synchronise before and after each."""
        out = self.new_out()
        if jt_prev is None:
            jt_prev = self.tru.eval_batch(self.Zd[par], want=("jac",))["jac"]
        torch.cuda.synchronize()
        Z = self.Zd[par]
        steps = [
            lambda: self.blk.eval_batch(Z, out=out["eb"]),
            lambda: self.tru.eval_products_batch(Z, w=out["eb"]["grad"], y=out["eb"]["g"], want=("f", "g"), out=out["pr"]),
            lambda: self.tru.eval_hessian_batch(Z, self.lamd, sigma=self.sigmad, out=out["h"]),
            lambda: self.tru.eval_hessian_product_batch(Z, self.lamd, out["pr"]["jty"], sigma=self.sigmad, out=out["hv"]),
            lambda: self.tru.kkt_solve_batch(out["h"], jt_prev, self.dcd, out["hv"], out["pr"]["jw"], sx=self.sxd,
                                             out=out["kkt"]),
            lambda: self.tru.eval_batch(Z, out=out["jt"]),
            lambda: self.blk.eval_ragged(self.rag_index, {"Z": Z.view(-1), **out["rag"]}, self.rag_off),
            lambda: self.kin.eval_batch(Z, out=out["kin"]),
        ]
        for s in steps:
            s()
            torch.cuda.synchronize()
        out["jt_prev"] = jt_prev.clone()
        return out

    def check_reference(self, par):
        """The one-at-a-time results against their references, on three rows."""
        ref, Z, p = self.ref[par], self.Z[par], self.p
        rows = [0, self.B // 2 + 1, self.B - 1]
        npy = lambda t: t.cpu().numpy()
        o = Oracle(p)
        want = o.eval_batch(Z[rows])
        assert_same_bits(self.blk, {k: npy(ref["eb"][k])[rows] for k in ALL}, want, f"{par}: block ")
        want_t = o.eval_batch(Z[rows], pattern="true")
        assert_same_bits(self.tru, {k: npy(ref["jt"][k])[rows] for k in ALL}, want_t, f"{par}: true ")
        # kinematic handle: its own rows have the oracle's bits (sqrt, IEEE division), the rest is the plain handle's
        n, m, nnz = p.n_nlp, p.m_nlp, self.blk.nnz
        want_k = Oracle(p, kinematics=True).eval_batch(Z[rows])
        kg, kj = npy(ref["kin"]["g"])[rows], npy(ref["kin"]["jac"])[rows]
        kin_j = self.kin.jacobian_structure_arrays()[0] > m
        assert np.array_equal(kg[:, m:], want_k["g"][:, m:]) and np.array_equal(kj[:, kin_j], want_k["jac"][:, kin_j])
        assert torch.equal(ref["kin"]["g"][:, :m], ref["eb"]["g"])
        assert torch.equal(ref["kin"]["jac"][:, ~torch.from_numpy(kin_j).cuda()], ref["eb"]["jac"])
        assert torch.equal(ref["kin"]["f"], ref["eb"]["f"]) and torch.equal(ref["kin"]["grad"], ref["eb"]["grad"])
        # ragged rows are the strided evaluation's rows (problem b at row b of the flat arrays)
        assert torch.equal(ref["rag"]["f"], ref["eb"]["f"])
        assert torch.equal(ref["rag"]["g"].view(self.B, m), ref["eb"]["g"])
        assert torch.equal(ref["rag"]["jac"].view(self.B, nnz), ref["eb"]["jac"])
        # products: the fold of the materialised SPARSE_TRUE values; f and g are the evaluator's
        assert torch.equal(ref["pr"]["f"], ref["jt"]["f"]) and torch.equal(ref["pr"]["g"], ref["jt"]["g"])
        jr, jc = self.tru.jacobian_structure_arrays()
        hr, hc = self.tru.hessian_structure_arrays()
        vals, w, y = npy(ref["jt"]["jac"]), npy(ref["eb"]["grad"]), npy(ref["eb"]["g"])
        jw, jty, H, hv = npy(ref["pr"]["jw"]), npy(ref["pr"]["jty"]), npy(ref["h"]), npy(ref["hv"])
        for b in rows[:2]:
            assert np.array_equal(jw[b], fold_rows(jr, jc, vals[b], w[b], m)), b
            assert np.array_equal(jty[b], fold_rows(jr, jc, vals[b], y[b], n, transpose=True)), b
            mr, mc, mv = mirrored(hr, hc, H[b])
            assert np.array_equal(hv[b], fold_rows(mr, mc, mv, jty[b], n)), b
        b = rows[1]
        hw = o.hess_lagrangian_dense(Z[b], self.sigma[b], self.lam[b])[hr - 1, hc - 1]
        assert np.abs(H[b] - hw).max() <= 1e-12 * max(1.0, np.abs(hw).max())
        # KKT solve: status 0 everywhere, and the step solves the assembled system
        px, pl, st = (npy(t) for t in ref["kkt"])
        assert (st == 0).all()
        jp = npy(ref["jt_prev"])
        for b in rows[:2]:
            K = kkt_ref.kkt_matrix((hr, hc), H[b], (jr, jc), jp[b], self.sx[b], self.dc[b])
            res, scale = kkt_ref.residual(K, px[b], pl[b], hv[b], jw[b])
            assert res <= 1e-12 * scale, (b, res, scale)

    def refs_without_prev(self, par):
        return {k: v for k, v in self.ref[par].items() if k != "jt_prev"}


def rig(ieee_div=False):
    if ieee_div not in _rigs:
        _rigs[ieee_div] = Rig(ieee_div)
    return _rigs[ieee_div]


@pytest.mark.parametrize("ieee_div", [False, True])
def test_mixed_families_on_one_stream(ieee_div):
    """The eight families queued back to back on one stream with no host synchronisation, four rounds alternating
    the two input sets, each round's outputs snapshotted by torch copies on the same stream.  Under QLNLP_IEEE_DIV
    every one-at-a-time result must also equal the default handles' bits: the reciprocal-FMA division is verified to
    round correctly, so the IEEE-division kernels (the only run of eval_prod_kernel<false>, hess_kernel<false> and
    hess_prod_kernel<false>) must agree with it everywhere."""
    r = rig(ieee_div)
    if ieee_div:
        d = rig(False)
        for par in (0, 1):
            _assert_equal_tree(r.refs_without_prev(par), d.refs_without_prev(par), f"IEEE division, inputs {par}")
    out = r.new_out()
    snaps = []
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        out["jt"]["jac"].copy_(r.ref[1]["jt"]["jac"])     # the Jacobian the first round's KKT solve reads
        for rnd in range(4):
            par = rnd % 2
            r.chain(par, out, out["jt"]["jac"])
            snaps.append((par, _clone_tree(out)))
    s.synchronize()
    for rnd, (par, snap) in enumerate(snaps):
        _assert_equal_tree(snap, r.refs_without_prev(par), f"round {rnd}")


def test_concurrent_streams_of_one_handle():
    """The same launches each on a stream of its own at once (the SPARSE_TRUE handle's products, Hessian, Hessian
    product, KKT solve and evaluation on five streams; the SPARSE_BLOCK handle's evaluation and ragged launch on two
    more; the kinematic handle on an eighth), beside one long g-only grid (B = 65,536) on a ninth stream; then the
    SPARSE_BLOCK and SPARSE_TRUE handles alternating on one stream.  Two rounds, inputs alternating."""
    r = rig(False)
    B = 256
    sub = lambda t: t[:B]
    streams = _RawStreams(10)
    try:
        st = streams.streams
        outs, long_out = [], []
        Zlong = [z[:B].repeat(65536 // B, 1) for z in r.Zd]
        torch.cuda.synchronize()
        for rnd in range(2):
            par = rnd % 2
            ref = r.ref[par]
            Z = sub(r.Zd[par])
            o = {"eb": _nan_tree({k: sub(v) for k, v in ref["eb"].items()}),
                 "pr": _nan_tree({k: sub(v) for k, v in ref["pr"].items()}),
                 "h": _nan_like(sub(ref["h"])), "hv": _nan_like(sub(ref["hv"])),
                 "kkt": _nan_tree(tuple(sub(t) for t in ref["kkt"])),
                 "jt": _nan_tree({k: sub(v) for k, v in ref["jt"].items()}),
                 "rag": {"g": torch.full((B * r.p.m_nlp,), float("nan"), dtype=torch.float64, device="cuda")},
                 "kin": _nan_tree({k: sub(v) for k, v in ref["kin"].items()})}
            lo = torch.full((65536, r.p.m_nlp), float("nan"), dtype=torch.float64, device="cuda")
            index = torch.arange(B, dtype=torch.int64, device="cuda")
            torch.cuda.synchronize()
            with torch.cuda.stream(st[0]):
                r.blk.eval_batch(Zlong[par], want=("g",), out={"g": lo})
            launches = [
                lambda: r.tru.eval_products_batch(Z, w=sub(ref["eb"]["grad"]), y=sub(ref["eb"]["g"]), want=("f", "g"),
                                                  out=o["pr"]),
                lambda: r.tru.eval_hessian_batch(Z, sub(r.lamd), sigma=sub(r.sigmad), out=o["h"]),
                lambda: r.tru.eval_hessian_product_batch(Z, sub(r.lamd), sub(ref["pr"]["jty"]), sigma=sub(r.sigmad),
                                                         out=o["hv"]),
                lambda: r.tru.kkt_solve_batch(sub(ref["h"]), sub(ref["jt_prev"]), sub(r.dcd), sub(ref["hv"]),
                                              sub(ref["pr"]["jw"]), sx=sub(r.sxd), out=o["kkt"]),
                lambda: r.tru.eval_batch(Z, out=o["jt"]),
                lambda: r.blk.eval_batch(Z, out=o["eb"]),
                lambda: r.blk.eval_ragged(index, {"Z": Z.reshape(-1), "g": o["rag"]["g"]}, {**r.rag_off}),
                lambda: r.kin.eval_batch(Z, out=o["kin"]),
            ]
            for i, launch in enumerate(launches):
                with torch.cuda.stream(st[1 + i]):
                    launch()
            # two handles on one stream: SPARSE_BLOCK and SPARSE_TRUE evaluations alternating
            with torch.cuda.stream(st[9]):
                two = [_nan_tree({k: sub(v) for k, v in ref[key].items()}) for key in ("eb", "jt", "eb", "jt")]
                for j, t in enumerate(two):
                    (r.blk if j % 2 == 0 else r.tru).eval_batch(Z, out=t)
            torch.cuda.synchronize()
            outs.append((par, o, two))
            long_out.append((par, lo))
        for par, o, two in outs:
            ref = r.ref[par]
            want = {"eb": {k: sub(v) for k, v in ref["eb"].items()}, "pr": {k: sub(v) for k, v in ref["pr"].items()},
                    "h": sub(ref["h"]), "hv": sub(ref["hv"]), "kkt": tuple(sub(t) for t in ref["kkt"]),
                    "jt": {k: sub(v) for k, v in ref["jt"].items()},
                    "rag": {"g": sub(ref["eb"]["g"]).reshape(-1)},
                    "kin": {k: sub(v) for k, v in ref["kin"].items()}}
            _assert_equal_tree(o, want, f"inputs {par}")
            for j, t in enumerate(two):
                _assert_equal_tree(t, want["eb" if j % 2 == 0 else "jt"], f"one stream, two handles, launch {j}")
        for par, lo in long_out:
            _assert_equal_tree(lo, r.ref[par]["eb"]["g"][:B].repeat(65536 // B, 1), f"B = 65,536 g only, inputs {par}")
    finally:
        streams.close()


def _graph_body(r, par, out, tru=None, kin=None):
    """What each captured graph holds: a SPARSE_TRUE evaluation, a KKT solve on its Jacobian, a kinematic evaluation
    (by the rig's handles unless others are given)."""
    ref, tru, kin = r.ref[par], tru or r.tru, kin or r.kin
    tru.eval_batch(r.Zd[par], out=out["jt"])
    tru.kkt_solve_batch(ref["h"], out["jt"]["jac"], r.dcd, ref["hv"], ref["pr"]["jw"], sx=r.sxd, out=out["kkt"])
    kin.eval_batch(r.Zd[par], out=out["kin"])


def _graph_want(r, par):
    """The graph's results made alone: the KKT solve there reads the Jacobian of its own inputs."""
    ref = r.ref[par]
    kkt = r.tru.kkt_solve_batch(ref["h"], ref["jt"]["jac"], r.dcd, ref["hv"], ref["pr"]["jw"], sx=r.sxd)
    torch.cuda.synchronize()
    st = kkt[2].cpu().numpy()
    assert (st == 0).all()
    hr, hc = r.tru.hessian_structure_arrays()
    jr, jc = r.tru.jacobian_structure_arrays()
    for b in (0, r.B - 1):
        K = kkt_ref.kkt_matrix((hr, hc), ref["h"][b].cpu().numpy(), (jr, jc), ref["jt"]["jac"][b].cpu().numpy(),
                               r.sx[b], r.dc[b])
        res, scale = kkt_ref.residual(K, kkt[0][b].cpu().numpy(), kkt[1][b].cpu().numpy(), ref["hv"][b].cpu().numpy(),
                                      ref["pr"]["jw"][b].cpu().numpy())
        assert res <= 1e-12 * scale, (b, res, scale)
    return {"jt": ref["jt"], "kkt": tuple(t.clone() for t in kkt), "kin": ref["kin"]}


def _capture(r, pars, **handles):
    """One graph per input set in `pars`, captured by torch.cuda.graph without stream=: all on torch's one default
    capture stream.  That stream is used eagerly first (which also gives it the per-stream scratch that capture once
    required)."""
    graphs, outs = [], []
    for par in pars:
        g = torch.cuda.CUDAGraph()
        ctx = torch.cuda.graph(g)
        cap = torch.cuda.graph.default_capture_stream
        out = {"jt": _nan_tree(r.ref[par]["jt"]), "kkt": _nan_tree(r.ref[par]["kkt"]), "kin": _nan_tree(r.ref[par]["kin"])}
        cap.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(cap):
            _graph_body(r, par, out, **handles)
        cap.synchronize()
        with ctx:
            _graph_body(r, par, out, **handles)
        graphs.append(g)
        outs.append(out)
    return graphs, outs, torch.cuda.graph.default_capture_stream


def test_graph_replays():
    """Two graphs captured on the same stream, replayed concurrently on two streams (three rounds); then one of them
    replayed while eager work of the same handles runs on the capture stream."""
    r = rig(False)
    want = [_graph_want(r, par) for par in (0, 1)]
    graphs, outs, cap = _capture(r, (0, 1))
    s = [torch.cuda.Stream(), torch.cuda.Stream()]
    for rnd in range(3):
        for o in outs:
            _fill_nan(o)
        torch.cuda.synchronize()
        for i in (0, 1):
            with torch.cuda.stream(s[i]):
                graphs[i].replay()
        torch.cuda.synchronize()
        for i in (0, 1):
            _assert_equal_tree(outs[i], want[i], f"concurrent replay {rnd}, graph {i}")
    # one replay beside eager work of the same handles on the capture stream
    for rnd in range(2):
        _fill_nan(outs[0])
        eager = {"jt": _nan_tree(r.ref[1]["jt"]), "kkt": _nan_tree(r.ref[1]["kkt"]), "kin": _nan_tree(r.ref[1]["kin"])}
        torch.cuda.synchronize()
        with torch.cuda.stream(s[0]):
            graphs[0].replay()
        with torch.cuda.stream(cap):
            _graph_body(r, 1, eager)
        torch.cuda.synchronize()
        _assert_equal_tree(outs[0], want[0], f"replay beside eager work {rnd}")
        _assert_equal_tree(eager, want[1], f"eager work beside a replay {rnd}")


def test_more_streams_than_the_counter_pool():
    """Fresh handles launch on the default stream and on the capture stream (a graph is captured there), then on 70
    fresh streams in turn with no synchronisation between them: more streams than the library's pool of 64 stream
    work counters, so the pool starts over at the 63rd and its counters go to new streams.  The graph is replayed
    right after the pool has started over, beside the streams that take the counters next (the second of them takes
    the capture stream's old counter).  Every result is checked."""
    r = rig(False)
    tru = ql.HybridNLP.from_problem(r.p, pattern="true", hessian=True)
    kin = ql.HybridNLP.from_problem(r.p, kinematics=True)
    B = 256
    sub = lambda t: t[:B]
    res = []

    def launch(par):
        ref = r.ref[par]
        o = {"jt": _nan_tree({k: sub(ref["jt"][k]) for k in ("f", "g")}),
             "kkt": _nan_tree(tuple(sub(t) for t in ref["kkt"])),
             "kin": _nan_tree({k: sub(ref["kin"][k]) for k in ("f", "g")})}
        tru.eval_batch(sub(r.Zd[par]), want=("f", "g"), out=o["jt"])
        tru.kkt_solve_batch(sub(ref["h"]), sub(ref["jt_prev"]), sub(r.dcd), sub(ref["hv"]), sub(ref["pr"]["jw"]),
                            sx=sub(r.sxd), out=o["kkt"])
        kin.eval_batch(sub(r.Zd[par]), want=("f", "g"), out=o["kin"])
        res.append((par, o))

    launch(0)                                             # the default stream: the handles' set-up
    torch.cuda.synchronize()
    want = _graph_want(r, 0)
    graphs, outs, cap = _capture(r, (0,), tru=tru, kin=kin)
    streams = _RawStreams(70)
    try:
        st = streams.streams
        torch.cuda.synchronize()
        for i in range(63):
            with torch.cuda.stream(st[i]):
                launch(i % 2)
        _fill_nan(outs[0])
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            graphs[0].replay()
        for i in range(63, 70):
            with torch.cuda.stream(st[i]):
                launch(i % 2)
        torch.cuda.synchronize()
        _assert_equal_tree(outs[0], want, "replay beside the streams that took the pool's counters over")
        for i, (par, o) in enumerate(res):
            ref = r.ref[par]
            w = {"jt": {k: sub(ref["jt"][k]) for k in ("f", "g")}, "kkt": tuple(sub(t) for t in ref["kkt"]),
                 "kin": {k: sub(ref["kin"][k]) for k in ("f", "g")}}
            _assert_equal_tree(o, w, f"launch {i}")
    finally:
        streams.close()


def test_kinematic_scratch_outlives_larger_eager_batches():
    """A kinematic evaluation captured at B = 600, then an eager one at B = 4,096 on the capture stream (a batch
    larger than any before it on that stream), then a replay: the graph's rows must not have moved under it."""
    r = rig(False)
    g = torch.cuda.CUDAGraph()
    ctx = torch.cuda.graph(g)
    cap = torch.cuda.graph.default_capture_stream
    out = _nan_tree(r.ref[0]["kin"])
    cap.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(cap):
        r.kin.eval_batch(r.Zd[0], out=out)
    cap.synchronize()
    with ctx:
        r.kin.eval_batch(r.Zd[0], out=out)
    big = torch.cat([r.Zd[1]] * 7)[:4096].contiguous()
    cap.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(cap):
        eager = r.kin.eval_batch(big)
    cap.synchronize()
    _fill_nan(out)
    torch.cuda.synchronize()
    g.replay()
    torch.cuda.synchronize()
    _assert_equal_tree(out, r.ref[0]["kin"], "replay after a larger eager batch")
    rep = lambda t: torch.cat([t] * 7)[:4096]
    _assert_equal_tree(eager, {k: rep(v) for k, v in r.ref[1]["kin"].items()}, "eager B = 4,096")


def _refused_in_capture(call):
    """`call` inside a capture must be refused with QLNLP_EINVAL and a message that says to warm the handle first;
    the capture itself must survive (a torch kernel captured beside the call replays)."""
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
    assert err is not None, "set-up inside a capture was not refused"
    assert err.code == qev.QLNLP_EINVAL, str(err)
    assert "warm the handle" in str(err) and "capture" in str(err), str(err)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(x, torch.ones_like(x))


def test_set_up_inside_a_capture_is_refused():
    """The first call of a fresh handle, the first kinematic evaluation, the first KKT solve and a ragged launch over
    a new set of classes need set-up (allocations, copies, a synchronise) that a capture cannot hold: each is refused
    cleanly, and once the same call has been made outside a capture it can be captured."""
    r = rig(False)
    p = r.p
    B = 8
    Z = r.Zd[0][:B]
    fresh = ql.HybridNLP.from_problem(p)
    _refused_in_capture(lambda: fresh.eval_batch(Z))
    # a kinematic handle whose device is bound (by a batched initial guess) but whose kinematic rows are not set up
    kin = ql.HybridNLP.from_problem(p, kinematics=True)
    x0 = torch.from_numpy(np.tile(p.x0, (B, 1))).cuda()
    kin.initial_guess_batch(x0)
    torch.cuda.synchronize()
    _refused_in_capture(lambda: kin.eval_batch(Z))
    # a SPARSE_TRUE handle that has evaluated but never solved
    tru = ql.HybridNLP.from_problem(p, pattern="true", hessian=True)
    ref = r.ref[0]
    tru.eval_batch(Z, want=("jac",))
    torch.cuda.synchronize()
    kkt = lambda: tru.kkt_solve_batch(ref["h"][:B], ref["jt"]["jac"][:B], r.dcd[:B], ref["hv"][:B],
                                      ref["pr"]["jw"][:B], sx=r.sxd[:B])
    _refused_in_capture(kkt)
    # ragged launches over classes (a single handle, then a pair) whose class table does not exist yet
    blk2 = ql.HybridNLP.from_problem(p)
    blk2.eval_batch(Z, want=("g",))
    torch.cuda.synchronize()
    index = torch.arange(B, dtype=torch.int64, device="cuda")
    off = {k: v[:B] for k, v in r.rag_off.items()}
    flat = lambda: {"Z": Z.reshape(-1), "g": torch.empty(B * p.m_nlp, dtype=torch.float64, device="cuda")}
    _refused_in_capture(lambda: blk2.eval_ragged(index, flat(), off))
    cls = torch.zeros(B, dtype=torch.int32, device="cuda")
    _refused_in_capture(lambda: ql.HybridNLP.eval_ragged_classes([blk2, r.blk], index, cls, flat(), off))
    # warmed outside a capture, every one of them can be captured, and the replay gives the eager bits
    calls = [lambda: fresh.eval_batch(Z), lambda: kin.eval_batch(Z), kkt,
             lambda: blk2.eval_ragged(index, flat(), off),
             lambda: ql.HybridNLP.eval_ragged_classes([blk2, r.blk], index, cls, flat(), off)]
    for c in calls:
        c()
    torch.cuda.synchronize()
    outs = {}
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        outs["fresh"] = fresh.eval_batch(Z)
        outs["kin"] = kin.eval_batch(Z)
        outs["kkt"] = kkt()
    _fill_nan(outs)
    g.replay()
    torch.cuda.synchronize()
    _assert_equal_tree(outs, {"fresh": {k: v[:B] for k, v in ref["eb"].items()},
                              "kin": {k: v[:B] for k, v in ref["kin"].items()},
                              "kkt": tuple(t[:B] for t in _graph_want(r, 0)["kkt"])}, "captured after warming")
