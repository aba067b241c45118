"""Parity of the CUDA path (through the C ABI) against the CPU oracle on the same seeded inputs.

Tolerance (BASELINE.json north_star): |a - b| <= 1e-14 + 1e-12 |b| in fp64; structure bit-exact.
f, g, grad and the Jacobian values are in fact expected to be BIT-IDENTICAL to the oracle (same operation order, no
FMA; the cost is accumulated knot by knot like costs.jl:9-15), except the 2N entries that go through sin/cos.
"Bit-identical" is a statement about the ORACLE: nothing in the reference pins grad_f!/jac_c! numerically, and the
oracle assumes ForwardDiff's dual product is un-fused (DESIGN.md section 2).
"""
import numpy as np
import pytest

from conftest import assert_parity, perturbed_batch
from oracle.oracle import Oracle
import quadruped_landing_b200 as ql

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def dflt():
    p = ql.default_problem()
    return p, ql.HybridNLP.from_problem(p), Oracle(p)


def assert_same_bits(nlp, got, ref, what=""):
    """g / grad / jac must be bit-identical to the oracle (same operation order, no FMA) except where
    sin/cos enter (body-clearance rows, constraints.jl:109,270-272): CUDA's libm and glibc may differ in
    the last ulp there, so those entries are held to the stated tolerance instead."""
    N = nlp.N
    for k in ("grad", "g", "jac"):
        if k not in got:
            continue
        a, b = got[k], ref[k]
        assert_parity(a, b, f"{what}{k}")
        if k == "g":
            trig = np.zeros(nlp.m_nlp, dtype=bool)
            trig[nlp.m_nlp - N:] = True
        elif k == "jac":
            rows, cols = nlp.jacobian_structure_arrays()        # of the handle's sparse pattern
            trig = (rows > nlp.m_nlp - N) & ((cols - 1) % 20 == 2)
        else:
            trig = np.zeros(nlp.n_nlp, dtype=bool)
        assert np.array_equal(a[..., ~trig], b[..., ~trig]), f"{what}{k}: bits differ outside the sin/cos entries"
        d = np.abs(a[..., trig] - b[..., trig])      # operands are O(1): a few ulp(1) at most
        assert d.size == 0 or d.max() <= 4 * np.finfo(np.float64).eps, f"{what}{k}: sin/cos entries differ by {d.max()}"
    if "f" in got:
        assert np.array_equal(got["f"], ref["f"]), f"{what}f: bits differ"


def _bases(p, golden):
    return [ql.initial_guess(p)] + [golden[f"data_{i}"] for i in range(1, 7)]


def _dev_eval(nlp, Z, **kw):
    # alternate between tightly packed rows (odd ld: cp.async staging) and rows padded to an even length
    # (16-byte aligned: one TMA bulk load per vector) so both input paths are exercised by every test
    _dev_eval.flip = not getattr(_dev_eval, "flip", False)
    if _dev_eval.flip:
        Zd = torch.zeros((Z.shape[0], Z.shape[1] + 1), dtype=torch.float64, device="cuda")[:, :Z.shape[1]]
        Zd.copy_(torch.from_numpy(Z))
    else:
        Zd = torch.from_numpy(Z).cuda()
    kw = {k: (torch.from_numpy(v).cuda() if isinstance(v, np.ndarray) else v) for k, v in kw.items()}
    out = nlp.eval_batch(Zd, **kw)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


def test_known_answers_through_the_gpu(dflt, golden):
    p, nlp, o = dflt
    z = golden["data_6"]
    # main.ipynb:710,712 (the same pins tests/test_oracle_kat.py holds for the oracle)
    f = nlp.eval_objective(z)
    assert f == 1.1608112892558562e+02               # main.ipynb:710, to the last bit (sequential accumulation)
    g = np.empty(nlp.m_nlp)
    nlp.eval_constraint(g, z)
    assert np.abs(g[:1032]).max() == 1.4928675395736724e-06
    grad = np.empty(nlp.n_nlp)
    nlp.eval_objective_gradient(grad, z)
    vals = np.empty(nlp.nnz)
    nlp.eval_constraint_jacobian(vals, z)
    assert_same_bits(nlp, {"g": g, "grad": grad, "jac": vals},
                     {"g": o.eval_c(z), "grad": o.grad_f(z), "jac": o.jac_c_sparse(z)})


def test_c2_batch_4096_against_oracle(dflt, golden):
    """SURVEY.md 8d C2: B=4096, Z_b = base[b mod 7] + 1e-2 xi_b, seed 4096, checked entry by entry."""
    p, nlp, o = dflt
    Z = perturbed_batch(p, _bases(p, golden), 4096, 1e-2, 4096)
    got = _dev_eval(nlp, Z)
    ref = o.eval_batch(Z)
    assert_same_bits(nlp, got, ref)      # stated tolerance everywhere + same bits outside sin/cos


def test_unperturbed_bases_exact_cancellation(dflt, golden):
    """At the reference trajectory the torque terms cancel exactly; parity must survive that."""
    p, nlp, o = dflt
    Z = np.stack(_bases(p, golden))
    got = _dev_eval(nlp, Z)
    ref = o.eval_batch(Z)
    assert_same_bits(nlp, got, ref)


@pytest.mark.parametrize("N,kt,im", [(31, 11, 1), (41, 14, 2), (61, 21, 2), (81, 27, 1), (101, 34, 2), (121, 41, 1),
                                     (2, 1, 1), (3, 2, 2), (33, 33, 1), (33, 1, 2), (64, 32, 1), (65, 2, 2)])
def test_other_horizons_and_schedules(N, kt, im):
    """SURVEY.md 8d C4 classes (varying horizon / contact schedule) plus edge cases of the pass/segment logic."""
    p = ql.build_problem(N=N, k_trans=kt, init_mode=im)
    nlp, o = ql.HybridNLP.from_problem(p), Oracle(p)
    base = ql.initial_guess(p) if kt > 1 else np.zeros(p.n_nlp)
    Z = perturbed_batch(p, [base], 300, 1e-2, 7)
    got = _dev_eval(nlp, Z)
    ref = o.eval_batch(Z)
    assert_same_bits(nlp, got, ref)


def test_per_evaluation_boundary_states(dflt):
    """SURVEY.md 8d C3: every problem of a sweep has its own x0 (drop height / pitch)."""
    p, nlp, o = dflt
    B = 64
    rng = np.random.default_rng(5)
    x0 = np.stack([ql.default_states(p.model, h_drop=h, theta0_deg=t)[0]
                   for h, t in zip(np.linspace(0.25, 3.0, B), np.linspace(-40, -5, B))])
    xf = np.tile(p.xf, (B, 1)) + 1e-3 * rng.standard_normal((B, 15))
    Z = perturbed_batch(p, [ql.initial_guess(p)], B, 1e-2, 11)
    got = _dev_eval(nlp, Z, x0=x0, xf=xf)
    ref = o.eval_batch(Z, x0=x0, xf=xf)
    assert_same_bits(nlp, got, ref)


def test_host_pointer_batch_and_partial_outputs(dflt, golden):
    p, nlp, o = dflt
    Z = perturbed_batch(p, _bases(p, golden), 1300, 1e-2, 13)      # > 2 pipeline chunks, ragged tail
    got = nlp.eval_batch_host(Z)
    ref = o.eval_batch(Z)
    assert_same_bits(nlp, got, ref)
    only = nlp.eval_batch_host(Z[:5], want=("g",))
    assert set(only) == {"g"}
    assert_same_bits(nlp, only, {"g": ref["g"][:5]})
    only = nlp.eval_batch_host(Z[:5], want=("f", "grad"))
    assert_same_bits(nlp, only, {"grad": ref["grad"][:5], "f": ref["f"][:5]})


def test_both_input_staging_paths_agree(dflt, golden):
    """Z rows padded to an even length are fetched with one TMA bulk load, tightly packed rows with cp.async."""
    p, nlp, o = dflt
    Z = perturbed_batch(p, _bases(p, golden), 777, 1e-2, 31)
    packed = torch.from_numpy(Z).cuda()
    padded = torch.full((777, 1216), float("nan"), dtype=torch.float64, device="cuda")
    padded[:, :1215] = packed
    a = nlp.eval_batch(packed)
    b = nlp.eval_batch(padded[:, :1215])
    torch.cuda.synchronize()
    for k in ("f", "grad", "g", "jac"):
        assert torch.equal(a[k], b[k]), k
    assert_same_bits(nlp, {k: v.cpu().numpy() for k, v in b.items()}, o.eval_batch(Z))


def test_unaligned_jacobian_rows_take_the_plain_store_path(dflt, golden):
    """nnz_block is odd: tightly packed rows are only 8-byte aligned, so the TMA path must not be used."""
    p, nlp, o = dflt
    Z = perturbed_batch(p, _bases(p, golden), 33, 1e-2, 17)
    Zd = torch.from_numpy(Z).cuda()
    jac = torch.empty((33, nlp.nnz_block), dtype=torch.float64, device="cuda")      # ld = 32161 (odd)
    out = nlp.eval_batch(Zd, want=("jac",), out={"jac": jac})
    torch.cuda.synchronize()
    assert_same_bits(nlp, {"jac": out["jac"].cpu().numpy()}, o.eval_batch(Z, want=("jac",)))


def test_dense_mode_is_the_references_matrix(golden):
    p = ql.default_problem()
    nlp = ql.HybridNLP.from_problem(p, use_sparse_jacobian=False)
    o = Oracle(p)
    z = golden["data_3"]
    vec = np.full(nlp.nnz, np.nan)
    nlp.eval_constraint_jacobian(vec, z)
    jac = vec.reshape(nlp.n_nlp, nlp.m_nlp).T               # reshape(vec, m_nlp, n_nlp), moi.jl:20
    assert_parity(jac, o.jac_c_dense(z), "dense jac")
    rows, cols = ql.HybridNLP.from_problem(p).jacobian_structure_arrays()
    mask = np.zeros(jac.shape, dtype=bool)
    mask[rows - 1, cols - 1] = True
    assert not jac[~mask].any()                             # everything the reference leaves unassigned is 0


def test_large_batch_properties():
    """At full size (SURVEY.md 8d C3: 65,536 problems) the oracle is too slow to compare everything, so
    check size-independent properties: constant entries of the value stream, rows that copy Z, and
    position independence (a vector evaluates to the same bits wherever it sits in the batch)."""
    p = ql.default_problem()
    nlp, o = ql.HybridNLP.from_problem(p), Oracle(p)
    B = 65536
    small = perturbed_batch(p, [ql.initial_guess(p)], 256, 5e-2, 2 ** 20)
    Zd = torch.from_numpy(small).cuda().repeat(B // 256, 1)
    out = nlp.eval_batch(Zd)
    torch.cuda.synchronize()
    ref = o.eval_batch(small)
    for k in ("grad", "g", "jac"):
        t = out[k].view(B // 256, 256, -1)
        assert bool((t == t[0:1]).all()), k                 # position independence
        assert_same_bits(nlp, {k: t[0].cpu().numpy()}, {k: ref[k]})
    f = out["f"].view(B // 256, 256)
    assert bool((f == f[0:1]).all())
    g = out["g"]
    assert bool((g[:, 929:990] == Zd[:, 4::20]).all())      # contact-first rows are y1_k
    rows, cols = nlp.jacobian_structure_arrays()
    const = np.nonzero((rows >= 30) & (rows <= 929) & (((rows - 30) // 15 + 1) * 20 < cols))[0]   # -I blocks
    jc = out["jac"][:, torch.from_numpy(const).cuda()]
    expect = torch.from_numpy(np.where((rows[const] - 30) % 15 == (cols[const] - 1) % 20, -1.0, 0.0)).cuda()
    assert bool((jc == expect).all())


def test_c3_sweep_65536_problems_with_their_own_initial_state():
    """SURVEY.md 8d C3: 256 drop heights x 256 initial pitches, per-problem x0, guesses built on the device,
    all four outputs, then Z += 1e-3 xi for 3 'iterations'.  A strided sample is checked against the oracle."""
    p = ql.default_problem()
    nlp, o = ql.HybridNLP.from_problem(p), Oracle(p)
    x0 = ql.sweep_initial_states(p.model, np.linspace(0.25, 3.0, 256), np.linspace(-40.0, -5.0, 256))
    x0d = torch.from_numpy(x0).cuda()
    Z = ql.initial_guess_batch(p, x0d, xp=torch)
    assert Z.shape == (65536, 1215) and Z.is_cuda
    gen = torch.Generator(device="cuda").manual_seed(3)
    sample = np.arange(0, 65536, 257)
    out = None
    for it in range(3):
        out = nlp.eval_batch(Z, x0=x0d, out=out)
        torch.cuda.synchronize()
        Zs = Z[torch.from_numpy(sample).cuda()].cpu().numpy()
        ref = o.eval_batch(Zs, x0=x0[sample])
        got = {k: v[torch.from_numpy(sample).cuda()].cpu().numpy() for k, v in out.items()}
        assert_same_bits(nlp, got, ref, f"iter {it}: ")
        # init rows are Z[x_1] - x0 for every problem (constraints.jl:149)
        assert bool((out["g"][:, :15] == Z[:, :15] - x0d).all())
        Z = Z + 1e-3 * torch.randn(Z.shape, generator=gen, device="cuda", dtype=torch.float64)


def test_c4_ragged_batch_of_mixed_horizons():
    """SURVEY.md 8d C4: (N, k_trans) in 6 classes x init_mode in {1, 2}, uniformly mixed, flat arrays + offsets."""
    classes = [(N, kt, im) for (N, kt) in [(31, 11), (41, 14), (61, 21), (81, 27), (101, 34), (121, 41)] for im in (1, 2)]
    probs = [ql.build_problem(N=N, k_trans=kt, init_mode=im) for N, kt, im in classes]
    ev = ql.RaggedEvaluator(probs)
    rng = np.random.default_rng(7)
    B = 4096
    class_of = rng.integers(0, len(classes), size=B)
    off = ev.offsets(class_of)
    guesses = [ql.initial_guess(p) for p in probs]
    vecs = []
    for b in range(B):
        v = guesses[class_of[b]] + 1e-2 * rng.standard_normal(probs[class_of[b]].n_nlp)
        v[19::20] = np.clip(v[19::20], 1e-3, 2e-2)         # clip the h entries like the other configs
        vecs.append(v)
    Zf = ev.pack(class_of, vecs)                           # rows padded to an even length: all 16-byte aligned
    out = ev.eval(class_of, torch.from_numpy(Zf).cuda())
    torch.cuda.synchronize()
    oracles = [Oracle(p) for p in probs]
    for b in range(0, B, 37):
        c = class_of[b]
        e = ev.nlps[c]
        z = vecs[b]
        ref = oracles[c].eval_batch(z[None, :])
        got = {"f": out["f"][b:b + 1].cpu().numpy(),
               "grad": out["grad"][off["z_off"][b]:off["z_off"][b] + e.n_nlp].cpu().numpy()[None, :],
               "g": out["g"][off["g_off"][b]:off["g_off"][b] + e.m_nlp].cpu().numpy()[None, :],
               "jac": out["jac"][off["j_off"][b]:off["j_off"][b] + e.nnz_block].cpu().numpy()[None, :]}
        assert_same_bits(ev.nlps[c], got, ref, f"problem {b} class {classes[c]}: ")


def test_ragged_one_launch_equals_launch_per_class():
    """qlnlp_eval_ragged_classes (one launch, class records swapped per warp) against qlnlp_eval_ragged_device per class:
    identical bits, for a batch whose classes come in random order, including classes with a single problem."""
    classes = [(31, 11, 1), (2, 1, 2), (61, 21, 2), (121, 41, 1), (33, 33, 2), (65, 2, 1)]
    probs = [ql.build_problem(N=N, k_trans=kt, init_mode=im) for N, kt, im in classes]
    ev = ql.RaggedEvaluator(probs)
    rng = np.random.default_rng(11)
    B = 777
    class_of = rng.integers(0, len(classes), size=B)
    class_of[5] = 1
    guesses = [ql.initial_guess(p) if p.k_trans > 1 else np.zeros(p.n_nlp) for p in probs]
    vecs = []
    for c in class_of:
        v = guesses[c] + 1e-2 * rng.standard_normal(probs[c].n_nlp)
        v[19::20] = np.clip(v[19::20], 1e-3, 2e-2)
        vecs.append(v)
    Zd = torch.from_numpy(ev.pack(class_of, vecs)).cuda()
    one = {k: v.clone() for k, v in ev.eval(class_of, Zd).items() if isinstance(v, torch.Tensor)}
    torch.cuda.synchronize()
    assert ev.nlps[0].launch_info()["blocks"] > 0
    # the reference: one qlnlp_eval_ragged_device launch per class over that class's problems
    off = ev.offsets(class_of)
    doff = {k: torch.from_numpy(v).cuda() for k, v in off.items()}
    per = {"Z": Zd, **{k: torch.empty_like(one[k]) for k in ("f", "grad", "g", "jac")}}
    for c, nlp in enumerate(ev.nlps):
        nlp.eval_ragged(torch.from_numpy(np.nonzero(class_of == c)[0]).cuda(), per, doff, z_padded=True)
    torch.cuda.synchronize()
    for b in range(B):          # compare the rows themselves (the padding between rows is never written)
        e = ev.nlps[class_of[b]]
        for k, o, w in (("grad", "z_off", e.n_nlp), ("g", "g_off", e.m_nlp), ("jac", "j_off", e.nnz_block)):
            lo = int(off[o][b])
            assert torch.equal(one[k][lo:lo + w], per[k][lo:lo + w]), (b, k)
    assert torch.equal(one["f"], per["f"])
    # partial outputs through the single launch
    only = ev.eval(class_of, Zd, want=("g",))
    torch.cuda.synchronize()
    for b in range(0, B, 50):
        lo, w = int(off["g_off"][b]), ev.nlps[class_of[b]].m_nlp
        assert torch.equal(only["g"][lo:lo + w], per["g"][lo:lo + w])


def test_c5_sized_shard_131072_per_gpu():
    """SURVEY.md 8d C5: 2^20 trajectories over 8 GPUs = 131,072 per GPU (33.7 GB of Jacobian values).  One shard
    is evaluated here; the result must not depend on the position in the batch, and a sample matches the oracle."""
    p = ql.default_problem()
    nlp, o = ql.HybridNLP.from_problem(p), Oracle(p)
    B = 131072
    small = perturbed_batch(p, [ql.initial_guess(p)], 512, 5e-2, 2 ** 20)
    Z = torch.from_numpy(small).cuda().repeat(B // 512, 1)
    out = nlp.eval_batch(Z, want=("g", "jac"))
    torch.cuda.synchronize()
    jac = out["jac"].view(B // 512, 512, -1)
    assert bool((jac[1:] == jac[:1]).all())
    assert_same_bits(nlp, {"jac": jac[0, :64].cpu().numpy(), "g": out["g"][:64].cpu().numpy()},
                     o.eval_batch(small[:64], want=("g", "jac")))


@pytest.mark.parametrize("N,kt,im", [(61, 21, 1), (33, 33, 2), (5, 2, 1), (64, 2, 2)])
def test_no_write_outside_the_rows(N, kt, im):
    """compute-sanitizer is closed on this pool, so out-of-bounds writes are hunted with canaries: every output
    row is padded (ld > width) and surrounded by guard rows filled with a sentinel that must survive."""
    p = ql.build_problem(N=N, k_trans=kt, init_mode=im)
    nlp = ql.HybridNLP.from_problem(p)
    B, guard, sentinel = 37, 3, -7.25
    Z = perturbed_batch(p, [ql.initial_guess(p) if kt > 1 else np.zeros(p.n_nlp)], B, 1e-2, 5)
    widths = {"grad": nlp.n_nlp, "g": nlp.m_nlp, "jac": nlp.nnz_block}
    for pad in (2, 3):                                     # even ld (TMA path when width is even too) and odd ld
        big, views = {}, {}
        for k, w in widths.items():
            big[k] = torch.full((B + 2 * guard, w + pad), sentinel, dtype=torch.float64, device="cuda")
            views[k] = big[k][guard:guard + B, :w]
        fbig = torch.full((B + 2 * guard,), sentinel, dtype=torch.float64, device="cuda")
        views["f"] = fbig[guard:guard + B]
        out = nlp.eval_batch(torch.from_numpy(Z).cuda(), out=dict(views))
        torch.cuda.synchronize()
        for k, w in widths.items():
            assert bool((big[k][:guard] == sentinel).all()) and bool((big[k][guard + B:] == sentinel).all()), k
            assert bool((big[k][:, w:] == sentinel).all()), k
            assert not bool((out[k] == sentinel).any()), k
        assert bool((fbig[:guard] == sentinel).all()) and bool((fbig[guard + B:] == sentinel).all())


@pytest.mark.parametrize("N,kt,im,B", [(61, 21, 1, 2048), (61, 21, 2, 300), (31, 11, 1, 300), (121, 41, 2, 300),
                                       (2, 1, 1, 40), (3, 2, 2, 40), (33, 33, 1, 100), (33, 1, 2, 100), (65, 2, 2, 100)])
def test_sparse_true_pattern(N, kt, im, B):
    """QLNLP_JAC_SPARSE_TRUE: only structural non-zeros (4,840 values at the default instance)."""
    p = ql.build_problem(N=N, k_trans=kt, init_mode=im)
    nlp, o = ql.HybridNLP.from_problem(p, pattern="true"), Oracle(p)
    base = ql.initial_guess(p) if kt > 1 else np.zeros(p.n_nlp)
    Z = perturbed_batch(p, [base], B, 1e-2, 21)
    got = _dev_eval(nlp, Z)
    ref = o.eval_batch(Z, pattern="true")
    assert got["jac"].shape == (B, o.nnz_true)
    assert_same_bits(nlp, got, ref)
    host = nlp.eval_batch_host(Z[:17])
    assert_same_bits(nlp, host, {k: v[:17] for k, v in ref.items()})
    vals = np.empty(nlp.nnz)
    nlp.eval_constraint_jacobian(vals, Z[0])                      # the MOI callback in SPARSE_TRUE order
    assert_same_bits(nlp, {"jac": vals}, {"jac": ref["jac"][0]})


def test_host_batch_compact_transfer_rebuilds_exact_rows(golden):
    """For host-pointer batches of >= 64 evaluations only the value-dependent Jacobian entries cross PCIe and host
    threads assemble the caller's rows from the constant image of the pattern: the rows must be identical to the
    device-resident result, including every zero, for B below / above the threshold and across chunk boundaries."""
    p = ql.default_problem()
    nlp = ql.HybridNLP.from_problem(p)
    Z = perturbed_batch(p, [ql.initial_guess(p)] + [golden[f"data_{i}"] for i in range(1, 7)], 1100, 1e-2, 99)
    dev = _dev_eval(nlp, Z)
    for B in (1, 63, 64, 256, 257, 512, 513, 1100):
        out = {"jac": np.full((B, nlp.nnz_block), np.nan)}
        host = nlp.eval_batch_host(Z[:B], out=out)
        for k in ("f", "grad", "g", "jac"):
            assert np.array_equal(host[k], dev[k][:B]), (B, k)
    # registered output rows: constant image written once, then only the lines that change -- three consecutive
    # calls with different Z (and a sub-range of the registered rows) must each give the device rows exactly
    jac = np.full((1100, nlp.nnz_block), np.nan)
    nlp.register_host_output(jac)
    before = nlp.host_path_info()
    for rep, (lo, hi) in enumerate([(0, 1100), (0, 1100), (100, 900)]):
        Zr = perturbed_batch(p, [golden[f"data_{1 + rep}"]], 1100, 2e-2, 500 + rep)
        devr = _dev_eval(nlp, Zr)
        host = nlp.eval_batch_host(Zr[lo:hi], out={"jac": jac[lo:hi]})
        assert np.array_equal(jac[lo:hi], devr["jac"][lo:hi]), rep
        assert np.array_equal(host["g"], devr["g"][lo:hi]) and np.array_equal(host["f"], devr["f"][lo:hi])
    after = nlp.host_path_info()
    lines = after["lines_written"] - before["lines_written"]
    assert lines <= (1100 + 1100 + 800) * 1800 < 3000 * after["lines_per_row"] / 2     # the touched lines only (<= 1742 per row, any alignment)
    nlp.unregister_host_output(jac)
    host = nlp.eval_batch_host(Z[:300], out={"jac": jac[:300]})
    assert np.array_equal(jac[:300], dev["jac"][:300])
    # SPARSE_TRUE rows take the same route
    nlp_t = ql.HybridNLP.from_problem(p, pattern="true")
    devt = _dev_eval(nlp_t, Z[:700])
    jt = np.full((700, nlp_t.nnz), np.nan)
    host = nlp_t.eval_batch_host(Z[:700], out={"jac": jt})
    assert np.array_equal(jt, devt["jac"])
    nlp_t.register_host_output(jt)
    Zr = perturbed_batch(p, [golden["data_2"]], 700, 2e-2, 77)
    nlp_t.eval_batch_host(Zr, out={"jac": jt})
    assert np.array_equal(jt, _dev_eval(nlp_t, Zr)["jac"])
    # the same through a DENSE handle (batches use SPARSE_BLOCK) and with per-evaluation boundary states
    nlp_d = ql.HybridNLP.from_problem(p, use_sparse_jacobian=False)
    x0 = np.tile(p.x0, (200, 1)) + 1e-3
    h2 = nlp_d.eval_batch_host(Z[:200], x0=x0)
    d2 = _dev_eval(nlp, Z[:200], x0=x0)
    assert np.array_equal(h2["jac"], d2["jac"]) and np.array_equal(h2["g"], d2["g"])


def _random_problem(seed, N=37, kt=12, im=2):
    """A problem with nothing at its default: model constants, per-knot cost tables, boundary states."""
    rng = np.random.default_rng(seed)
    model = ql.PlanarQuadruped(g=-3.71 - rng.random(), mb=7.3 + rng.random(), mf=0.23 + 0.1 * rng.random(),
                               lb=0.61 + 0.1 * rng.random(), l1=0.3, l2=0.2)
    obj = [ql.LQRCost(rng.uniform(0, 20, 15), rng.uniform(0, 1, 5), rng.normal(size=15), rng.normal(size=5) * 30)
           for _ in range(N)]
    return ql.ProblemData.from_costs(model, obj, im, kt, N, rng.normal(size=15), rng.normal(size=15))


@pytest.mark.parametrize("ieee_div", [False, True])
def test_non_default_model_and_cost_tables(ieee_div, monkeypatch):
    """Per-knot random Q/R/q/r/c and non-default model constants; both division instantiations of the kernel
    (reciprocal-FMA and IEEE) must give the oracle's bits."""
    if ieee_div:
        monkeypatch.setenv("QLNLP_IEEE_DIV", "1")
    p = _random_problem(17)
    nlp, o = ql.HybridNLP.from_problem(p), Oracle(p)
    rng = np.random.default_rng(18)
    Z = rng.normal(size=(500, p.n_nlp))
    Z[:, 19::20] = rng.uniform(1e-3, 2e-2, size=(500, p.N - 1))
    got = _dev_eval(nlp, Z)
    assert_same_bits(nlp, got, o.eval_batch(Z))
    nlp_t = ql.HybridNLP.from_problem(p, pattern="true")
    assert_same_bits(nlp_t, _dev_eval(nlp_t, Z[:100]), o.eval_batch(Z[:100], pattern="true"))


def test_non_finite_inputs_do_not_crash_and_stay_local(dflt):
    """The reference does no checks; NaN/Inf propagate.  Here they propagate through every operation that is kept;
    structurally zero Jacobian entries stay 0 (the reference would produce NaN there: 0*NaN).  Other evaluations
    of the batch are unaffected."""
    p, nlp, o = dflt
    Z = perturbed_batch(p, [ql.initial_guess(p)], 8, 1e-2, 3)
    Z[3, 20 * 10 + 1] = np.nan          # yb of knot 11
    Z[5, 20 * 40 + 16] = np.inf         # F1y of knot 41
    got = _dev_eval(nlp, Z)
    ref = o.eval_batch(Z)
    clean = [0, 1, 2, 4, 6, 7]
    assert_same_bits(nlp, {k: v[clean] for k, v in got.items()}, {k: v[clean] for k, v in ref.items()})
    assert np.isnan(got["f"][3]) and np.isnan(got["g"][3]).any() and not np.isfinite(got["f"][5])
    assert np.isfinite(got["g"][3]).sum() > 900          # only the rows that touch knot 10/11 are affected
    # B = 16,384: every resident warp evaluates several rows, clean ones after poisoned ones.  NaN or Inf in one entry
    # of every fifth row; the clean rows must be the bits of a batch of the clean rows alone, in every value stream
    # (none: no Jacobian; SPARSE_BLOCK; SPARSE_TRUE)
    B = 16384
    gen = torch.Generator(device="cuda").manual_seed(3)
    Zd = torch.from_numpy(ql.initial_guess(p)).cuda().repeat(B, 1)
    Zd += 1e-2 * torch.randn(Zd.shape, generator=gen, dtype=torch.float64, device="cuda")
    Zd[:, 19::20].clamp_(1e-3, 2e-2)
    bad = np.arange(4, B, 5)
    for j, b in enumerate(bad.tolist()):
        Zd[b, (20 * ((7 * j) % p.N) + j % 20) % p.n_nlp] = np.nan if j % 2 else np.inf
    clean = torch.from_numpy(np.setdiff1d(np.arange(B), bad)).cuda()
    true = ql.HybridNLP.from_problem(p, pattern="true")
    for h, want in ((nlp, ("f", "grad", "g")), (nlp, ("f", "grad", "g", "jac")), (true, ("f", "grad", "g", "jac"))):
        got, alone = h.eval_batch(Zd, want=want), h.eval_batch(Zd[clean], want=want)
        torch.cuda.synchronize()
        assert not bool(torch.isfinite(got["f"][torch.from_numpy(bad).cuda()]).any())
        for k in want:
            a, c = got[k][clean].contiguous(), alone[k].contiguous()
            assert bool(torch.isfinite(c).all()) and torch.equal(a.view(torch.int64), c.view(torch.int64)), (want, k)


def test_handles_of_different_sizes_coexist():
    """Kernel attributes are per function, not per handle: a small problem created later must not shrink the
    shared-memory limit a larger, older handle needs (regression test)."""
    big = ql.HybridNLP.from_problem(ql.build_problem(N=121, k_trans=41))
    zb = perturbed_batch(big.prob, [ql.initial_guess(big.prob)], 4, 1e-2, 1)
    a = _dev_eval(big, zb)
    small = ql.HybridNLP.from_problem(ql.build_problem(N=5, k_trans=3))
    _dev_eval(small, perturbed_batch(small.prob, [ql.initial_guess(small.prob)], 4, 1e-2, 1))
    b = _dev_eval(big, zb)
    assert np.array_equal(a["jac"], b["jac"])


def test_destroyed_handles_give_their_device_memory_back():
    """Every path allocates lazily inside the handle (device scratch, pinned stages, worker pool, single-evaluation
    cache, Hessian buffers): a create / use / destroy cycle must not leak device memory."""
    import gc
    p = ql.build_problem(N=21, k_trans=8)
    Z = perturbed_batch(p, [ql.initial_guess(p)], 700, 1e-2, 3)

    def cycle():
        for pattern in ("block", "true"):
            nlp = ql.HybridNLP.from_problem(p, pattern=pattern, hessian=True)
            nlp.eval_batch_host(Z)                                   # host path: lanes, stages, pool, row plan
            x = Z[0].copy()
            nlp.eval_objective(x)                                    # single-evaluation cache
            nlp.eval_hessian_lagrangian(np.empty(nlp.nnz_hess), x, 1.0, np.ones(nlp.m_nlp))
            _dev_eval(nlp, Z[:8])
            del nlp
        gc.collect()
        torch.cuda.synchronize()
        torch.cuda.empty_cache()

    cycle()                                                          # module load, context growth, allocator pools
    free0 = torch.cuda.mem_get_info()[0]
    for _ in range(5):
        cycle()
    free1 = torch.cuda.mem_get_info()[0]
    assert free0 - free1 < (8 << 20), f"{(free0 - free1) >> 20} MiB of device memory lost over 10 handles"


def test_solver_loop_on_the_gpu_evaluator():
    """SURVEY.md 8f N1: the solve() glue of moi.jl:46-103 driving the GPU evaluator through the four MOI callbacks
    with the SPARSE_TRUE structure (a few iterations; the callbacks must agree with the oracle at the iterate)."""
    import warnings
    from quadruped_landing_b200.solve import solve
    p = ql.build_problem(N=9, k_trans=4)
    nlp, o = ql.HybridNLP.from_problem(p, pattern="true"), Oracle(p)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        res = solve(ql.initial_guess(p), nlp, tol=1e-3, c_tol=1e-3, max_iter=5, backend="trust-constr")
    assert res.iterations == 5 and min(res.evals.values()) >= 5
    assert abs(res.objective - o.eval_f(res.x)) <= 1e-12 * max(1.0, abs(res.objective))
    vals = np.empty(nlp.nnz)
    nlp.eval_constraint_jacobian(vals, res.x)
    assert_same_bits(nlp, {"jac": vals}, {"jac": o.jac_c_sparse_true(res.x)})


def test_solver_loop_with_the_exact_hessian():
    """The same glue with :Hess switched on: the solver receives sigma Hess f + sum lam Hess g from the GPU."""
    import warnings
    from quadruped_landing_b200.solve import solve
    p = ql.build_problem(N=9, k_trans=4)
    nlp = ql.HybridNLP.from_problem(p, pattern="true", hessian=True)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        res = solve(ql.initial_guess(p), nlp, tol=1e-3, c_tol=1e-3, max_iter=5, backend="trust-constr")
    assert res.evals["hess"] >= 2 and np.isfinite(res.objective)


def test_randomised_stress_against_the_oracle():
    """tests/fuzz_gpu.py for 20 s: random classes (N in 2..121, any k_trans / init_mode), batch sizes 1..3000,
    paddings and alignments, output subsets, both sparse patterns, device and host entry points, canary rows.
    (Round 1: 1,176 cases in 150 s; round 2, with the added modes: 1,728 cases in 200 s, no failure.)"""
    import subprocess, sys, os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "tests", "fuzz_gpu.py"), "20", "7"], capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "0 failures" in r.stdout


def test_launches_can_be_captured_in_a_cuda_graph(dflt, golden):
    """The launch path makes no allocation or synchronising call (work counters come from a pre-zeroed pool and
    re-arm themselves), so a sequence of evaluations can be captured once and replayed as a CUDA graph."""
    p, nlp, o = dflt
    Z = perturbed_batch(p, _bases(p, golden), 600, 1e-2, 77)
    Zd = torch.zeros((600, 1216), dtype=torch.float64, device="cuda")[:, :1215]
    Zd.copy_(torch.from_numpy(Z))
    eager = {k: v.clone() for k, v in nlp.eval_batch(Zd).items()}
    torch.cuda.synchronize()
    out = {k: torch.zeros_like(v) for k, v in eager.items()}
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                       # warm the capture stream's work counter outside the capture
        nlp.eval_batch(Zd, out=out)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        nlp.eval_batch(Zd, out=out, want=("g", "jac"))
        nlp.eval_batch(Zd, out=out, want=("f", "grad"))
    for k in out:
        out[k].zero_()
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    for k in eager:
        assert torch.equal(out[k], eager[k]), k


def test_every_launcher_can_be_captured_in_a_cuda_graph(dflt, golden):
    """The products, the Hessian, the Hessian products, the KKT solve and a kinematic handle's evaluation launch
    through the same path as the plain evaluation: once the capture stream has been used (its work counter, the
    kinematic and KKT scratch), their launches can be captured into one graph whose replay equals the eager results."""
    p = dflt[0]
    nlp = ql.HybridNLP.from_problem(p, pattern="true", hessian=True)
    kin = ql.HybridNLP.from_problem(p, kinematics=True)
    B, n, m = 600, nlp.n_nlp, nlp.m_nlp
    rng = np.random.default_rng(12)
    cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    Z = cuda(perturbed_batch(p, _bases(p, golden), B, 1e-2, 12))
    lam, sigma = cuda(1e-4 * rng.standard_normal((B, m))), cuda(np.full(B, 1e-4))
    w, y, V = cuda(rng.standard_normal((B, n))), cuda(rng.standard_normal((B, m))), cuda(rng.standard_normal((B, n)))
    dc, sx = cuda(rng.uniform(1e-2, 1.0, (B, m))), cuda(rng.uniform(1.0, 10.0, (B, n)))
    r1, r2 = cuda(rng.standard_normal((B, n))), cuda(rng.standard_normal((B, m)))
    jac = nlp.eval_batch(Z, want=("jac",))["jac"]

    def run(out):
        nlp.eval_products_batch(Z, w=w, y=y, want=("f", "g"), out=out["prod"])
        nlp.eval_hessian_batch(Z, lam, sigma=sigma, out=out["hess"])
        nlp.eval_hessian_product_batch(Z, lam, V, sigma=sigma, out=out["hv"])
        nlp.kkt_solve_batch(out["hess"], jac, dc, r1, r2, sx=sx, out=out["kkt"])
        kin.eval_batch(Z, out=out["kin"])

    eager = {"prod": nlp.eval_products_batch(Z, w=w, y=y, want=("f", "g")), "hess": nlp.eval_hessian_batch(Z, lam, sigma=sigma),
             "hv": nlp.eval_hessian_product_batch(Z, lam, V, sigma=sigma), "kin": kin.eval_batch(Z)}
    eager["kkt"] = nlp.kkt_solve_batch(eager["hess"], jac, dc, r1, r2, sx=sx)
    torch.cuda.synchronize()
    assert not eager["kkt"][2].any()                    # every problem solved: the comparison covers real steps

    def like(t):                                        # same row stride as the library's outputs
        if t.dim() == 1:
            return torch.zeros_like(t)
        return torch.zeros((t.shape[0], t.stride(0)), dtype=t.dtype, device=t.device)[:, :t.shape[1]]

    out = {"prod": {k: like(v) for k, v in eager["prod"].items()}, "hess": like(eager["hess"]), "hv": like(eager["hv"]),
           "kkt": tuple(like(t) for t in eager["kkt"]), "kin": {k: like(v) for k, v in eager["kin"].items()}}
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                       # warm the capture stream outside the capture
        run(out)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        run(out)
    flat = lambda o: [*o["prod"].values(), o["hess"], o["hv"], *o["kkt"], *o["kin"].values()]
    for t in flat(out):
        t.zero_()
    for _ in range(2):
        g.replay()
    torch.cuda.synchronize()
    for i, (a, b) in enumerate(zip(flat(out), flat(eager))):
        assert torch.equal(a, b), i


def test_back_to_back_launches_respect_stream_order(dflt, golden):
    """Evaluations are launched with programmatic dependent launch: the next grid may be scheduled while the previous
    one drains, so the kernel itself has to wait for its predecessors before it touches data.  Queue, without any
    host synchronisation, (a) two evaluations of different inputs into the same outputs, (b) a torch kernel that
    reads the outputs between two evaluations, (c) a torch kernel that rewrites the inputs between two evaluations,
    many times over, and compare every snapshot with evaluations done one at a time."""
    p, nlp, o = dflt
    B = 1500                                          # a short grid: the hand-over between two grids is most of the run
    Za = perturbed_batch(p, _bases(p, golden), B, 1e-2, 5)
    Zb = perturbed_batch(p, _bases(p, golden), B, 2e-2, 6)
    pad = lambda Z: torch.zeros((B, 1216), dtype=torch.float64, device="cuda")[:, :1215].copy_(torch.from_numpy(Z))
    A, Bm = pad(Za), pad(Zb)
    ra = {k: v.clone() for k, v in nlp.eval_batch(A).items()}
    torch.cuda.synchronize()
    rb = {k: v.clone() for k, v in nlp.eval_batch(Bm).items()}
    torch.cuda.synchronize()
    delta = 1e-3 * torch.randn((B, 1215), dtype=torch.float64, device="cuda")
    W = A.clone()                                     # rewritten in place below
    Wp = pad(Za)
    Wp += delta
    rw = {k: v.clone() for k, v in nlp.eval_batch(Wp).items()}
    torch.cuda.synchronize()
    out = {k: torch.zeros_like(v) for k, v in ra.items()}
    snaps = []
    for _ in range(6):
        nlp.eval_batch(A, out=out)                    # (a)
        nlp.eval_batch(Bm, out=out)
        snaps.append(("b", {k: v.clone() for k, v in out.items()}))       # (b) torch reads what the 2nd launch wrote ...
        nlp.eval_batch(A, out=out)                    # ... and the 3rd overwrites it
        snaps.append(("a", {k: v.clone() for k, v in out.items()}))
        W.copy_(A)                                    # (c) torch rewrites the input of the next launch
        W += delta
        Wv = torch.zeros((B, 1216), dtype=torch.float64, device="cuda")[:, :1215]
        Wv.copy_(W)
        nlp.eval_batch(Wv, out=out)
        snaps.append(("w", {k: v.clone() for k, v in out.items()}))
    torch.cuda.synchronize()
    ref = {"a": ra, "b": rb, "w": rw}
    for tag, snap in snaps:
        for k in snap:
            assert torch.equal(snap[k], ref[tag][k]), (tag, k)


def test_eval_all_and_the_x_cache(dflt, golden):
    """qlnlp_eval_all = the four callbacks with one launch; the callbacks themselves are served from the last
    evaluation when x is unchanged (moi.jl:1-24 calls them one by one) -- and must notice an x changed IN PLACE."""
    p, nlp, o = dflt
    x = golden["data_4"].copy()
    f, grad, g, vals = np.empty(1), np.empty(nlp.n_nlp), np.empty(nlp.m_nlp), np.empty(nlp.nnz)
    nlp.eval_all(x, f, grad, g, vals)
    ref = o.eval_batch(x[None, :])
    assert f[0] == ref["f"][0]
    assert_same_bits(nlp, {"grad": grad, "g": g, "jac": vals}, {k: ref[k][0] for k in ("grad", "g", "jac")})
    # the four callbacks at the same x
    assert nlp.eval_objective(x) == f[0]
    g2 = np.empty(nlp.m_nlp)
    nlp.eval_constraint(g2, x)
    assert np.array_equal(g2, g)
    # x modified in place between two callbacks: the cache must not be used
    x[20 * 7 + 3] += 0.125
    x[19] = 0.0123
    nlp.eval_constraint(g2, x)
    ref2 = o.eval_batch(x[None, :])
    assert_same_bits(nlp, {"g": g2}, {"g": ref2["g"][0]})
    assert not np.array_equal(g2, g)
    v2 = np.empty(nlp.nnz)
    nlp.eval_constraint_jacobian(v2, x)
    assert_same_bits(nlp, {"jac": v2}, {"jac": ref2["jac"][0]})
    assert nlp.eval_objective(x) == ref2["f"][0]
    # cache off: same answers
    nlp.set_option("x_cache", 0)
    nlp.eval_objective_gradient(grad, x)
    assert_same_bits(nlp, {"grad": grad}, {"grad": ref2["grad"][0]})
    nlp.set_option("x_cache", 1)
    # partial outputs and the SPARSE_TRUE pattern
    nlp_t = ql.HybridNLP.from_problem(p, pattern="true")
    vt = np.empty(nlp_t.nnz)
    nlp_t.eval_all(x, vec=vt)
    assert_same_bits(nlp_t, {"jac": vt}, {"jac": o.jac_c_sparse_true(x)})


def test_calls_leave_the_current_device_alone(dflt):
    """A call on a handle must not change the thread's current CUDA device."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 devices")
    p, nlp, o = dflt
    nlp1 = ql.HybridNLP.from_problem(p, device=1)
    torch.cuda.set_device(0)
    nlp1.eval_objective(ql.initial_guess(p))
    assert torch.cuda.current_device() == 0
    del nlp1
    assert torch.cuda.current_device() == 0


@pytest.mark.parametrize("all_devices", [False, True], ids=["one_device", "all_devices"])
def test_multi_device_handle_shards_the_batch(golden, all_devices):
    """qlnlp_create_multi: one call spreads a host batch (contiguous shards, one pipeline per device) or launches one
    device-resident shard per GPU; results must equal the single-device ones bit for bit.  A multi-device handle over
    one device takes the same paths."""
    nd = torch.cuda.device_count() if all_devices else 1
    if all_devices and nd < 2:
        pytest.skip("needs at least 2 devices")
    p = ql.default_problem()
    one = ql.HybridNLP.from_problem(p)
    multi = ql.HybridNLP.from_problem(p, devices=list(range(nd)))
    Z = perturbed_batch(p, [ql.initial_guess(p)] + [golden[f"data_{i}"] for i in range(1, 7)], 1500 + nd + 1, 1e-2, 4)
    ref = _dev_eval(one, Z)
    host = multi.eval_batch_host(Z)
    for k in ("f", "grad", "g", "jac"):
        assert np.array_equal(host[k], ref[k]), k
    jac = np.full((Z.shape[0], multi.nnz_batch), np.nan)
    multi.register_host_output(jac)
    for rep in range(2):
        multi.eval_batch_host(Z, out={"jac": jac}, want=("jac",))
        assert np.array_equal(jac, ref["jac"])
    bounds = [ql.shard_bounds(Z.shape[0], nd, r) for r in range(nd)]
    Zs = [torch.from_numpy(Z[lo:hi]).to(f"cuda:{i}") for i, (lo, hi) in enumerate(bounds)]
    outs = multi.eval_batch_multi(Zs)
    multi.synchronize()
    for (lo, hi), out in zip(bounds, outs):
        for k in ("f", "grad", "g", "jac"):
            assert np.array_equal(out[k].cpu().numpy(), ref[k][lo:hi]), k
    assert torch.cuda.current_device() == 0
    with pytest.raises(ql.QlnlpError):
        multi.eval_batch(Zs[0])


@pytest.mark.parametrize("N,kt,im,B", [(61, 21, 1, 300), (61, 21, 2, 64), (31, 11, 2, 64), (2, 1, 1, 40), (2, 2, 2, 40),
                                       (33, 33, 1, 64), (33, 1, 2, 64), (65, 2, 1, 64), (121, 41, 1, 33)])
def test_lagrangian_hessian_against_the_oracle(N, kt, im, B):
    """SURVEY.md 8f N3 (no reference target: src/moi.jl:26-28): sigma Hess f + sum_r mu_r Hess g_r from the kernel
    generated out of second-order duals vs the oracle's dense second-order forward mode, batched and single."""
    p = ql.build_problem(N=N, k_trans=kt, init_mode=im)
    nlp, o = ql.HybridNLP.from_problem(p, hessian=True), Oracle(p)
    rng = np.random.default_rng(N + kt)
    base = ql.initial_guess(p) if kt > 1 else np.zeros(p.n_nlp)
    Z = perturbed_batch(p, [base], B, 5e-2, 9)
    mu = rng.standard_normal((B, p.m_nlp))
    sigma = rng.uniform(0.2, 2.0, size=B)
    rows, cols = nlp.hessian_structure_arrays()
    for padded in (False, True):
        if padded:
            Zd = torch.zeros((B, p.n_nlp + 1), dtype=torch.float64, device="cuda")[:, :p.n_nlp]
            Zd.copy_(torch.from_numpy(Z))
        else:
            Zd = torch.from_numpy(Z).cuda()
        H = nlp.eval_hessian_batch(Zd, torch.from_numpy(mu).cuda(), torch.from_numpy(sigma).cuda())
        torch.cuda.synchronize()
        H = H.cpu().numpy()
        for b in range(0, B, max(1, B // 6)):
            want = o.hess_lagrangian_dense(Z[b], sigma[b], mu[b])[rows - 1, cols - 1]
            tol = 1e-12 * max(1.0, np.abs(want).max())
            assert np.abs(H[b] - want).max() <= tol, (b, padded)
    # the MOI-style single call on host pointers
    vals = np.empty(nlp.nnz_hess)
    nlp.eval_hessian_lagrangian(vals, Z[1], sigma[1], mu[1])
    assert np.array_equal(vals, H[1])
    # position independence
    H2 = nlp.eval_hessian_batch(torch.from_numpy(Z[::-1].copy()).cuda(), torch.from_numpy(mu[::-1].copy()).cuda(),
                                torch.from_numpy(sigma[::-1].copy()).cuda())
    torch.cuda.synchronize()
    assert np.array_equal(H2.cpu().numpy()[::-1], H)


def test_empty_batches_are_not_an_error(dflt):
    """An empty shard (B = 0) returns empty outputs without touching the device (sharding with B < world size)."""
    p, nlp, o = dflt
    out = nlp.eval_batch(torch.empty((0, p.n_nlp), dtype=torch.float64, device="cuda"))
    assert out["jac"].shape == (0, nlp.nnz_block) and out["f"].shape == (0,)
    host = nlp.eval_batch_host(np.empty((0, p.n_nlp)))
    assert host["g"].shape == (0, nlp.m_nlp)


@pytest.mark.parametrize("N,kt,im", [(61, 21, 1), (31, 11, 2), (33, 33, 1), (5, 2, 2), (2, 2, 1)])
def test_initial_guess_kernel_matches_the_notebook_formula(N, kt, im):
    """SURVEY.md 8f N2: the sweep's guesses (main.ipynb:181-196) built by a CUDA kernel = the host formula, bit for bit,
    and the torch variant of problem.initial_guess_batch agrees with both."""
    p = ql.build_problem(N=N, k_trans=kt, init_mode=im)
    nlp = ql.HybridNLP.from_problem(p)
    x0 = ql.sweep_initial_states(p.model, np.linspace(0.25, 3.0, 13), np.linspace(-40.0, -5.0, 11))
    want = ql.initial_guess_batch(p, x0)
    x0d = torch.from_numpy(x0).cuda()
    got = nlp.initial_guess_batch(x0d)
    torch.cuda.synchronize()
    assert got.shape == want.shape and np.array_equal(got.cpu().numpy(), want)
    if kt > 1:
        # the eager-torch variant of problem.initial_guess_batch divides by multiplying with a reciprocal on the GPU:
        # equal to 1 ulp, not to the bit (the kernel above is the exact one)
        eager = ql.initial_guess_batch(p, x0d, xp=torch).cpu().numpy()
        assert np.abs(eager - want).max() <= 4 * np.finfo(np.float64).eps * max(1.0, np.abs(want).max())
    # the guess of the problem's own x0 is the class guess
    own = nlp.initial_guess_batch(torch.from_numpy(p.x0[None, :].copy()).cuda())
    assert np.array_equal(own.cpu().numpy()[0], ql.initial_guess(p))
