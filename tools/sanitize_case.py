"""Small cases that launch every kernel of the library once, written for compute-sanitizer (memcheck / racecheck /
synccheck).  The GPU pool of round 2 refuses compute-sanitizer runs, so here it only runs plainly with its own checks;
out-of-row writes are covered by the guard-band test (tests/test_gpu_parity.py::test_no_write_outside_the_rows).

SPARSE_BLOCK (bulk + plain store paths, per-evaluation x0), SPARSE_TRUE, the value-dependent stream of the host path,
a ragged mixed-class launch, the Lagrangian Hessian, the opt-in kinematic rows, the initial-guess kernel and the dense
scatter of the single-evaluation path."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import quadruped_landing_b200 as ql

rng = np.random.default_rng(0)
for (N, kt, im, B) in [(61, 21, 1, 40), (33, 33, 2, 9), (5, 2, 1, 3)]:
    p = ql.build_problem(N=N, k_trans=kt, init_mode=im)
    nlp = ql.HybridNLP.from_problem(p)
    Z = ql.initial_guess(p)[None, :] + 1e-2 * rng.standard_normal((B, p.n_nlp))
    Zd = torch.from_numpy(Z).cuda()
    x0 = torch.from_numpy(np.tile(p.x0, (B, 1))).cuda()
    out = nlp.eval_batch(Zd, x0=x0)
    jac = torch.empty((B, nlp.nnz_block), dtype=torch.float64, device="cuda")
    out2 = nlp.eval_batch(Zd, want=("jac",), out={"jac": jac})          # unaligned rows: plain store path
    nlp.eval_batch(Zd, want=("f", "grad", "g"))                         # the kernel without a Jacobian
    torch.cuda.synchronize()
    assert torch.equal(out["jac"], out2["jac"])
    h = nlp.eval_batch_host(Z)                                          # VALS stream + row assembly on the host
    assert np.array_equal(h["jac"], out["jac"].cpu().numpy())
    t = ql.HybridNLP.from_problem(p, pattern="true", hessian=True)
    ot = t.eval_batch(Zd)
    ht = t.eval_batch_host(Z)
    assert np.array_equal(ht["jac"], ot["jac"].cpu().numpy())
    mu = torch.from_numpy(rng.standard_normal((B, t.m_nlp))).cuda()
    t.eval_hessian_batch(Zd, mu)
    x = Z[0].copy()
    dense = ql.HybridNLP.from_problem(p, use_sparse_jacobian=False)
    vals = np.zeros(dense.nnz)
    dense.eval_constraint_jacobian(vals, x)                             # dense scatter kernel
    k = ql.HybridNLP.from_problem(p, kinematics=True)
    k.eval_batch(Zd)
    kv = np.empty(k.nnz); k.eval_constraint_jacobian(kv, x)
    guess = nlp.initial_guess_batch(x0)
    torch.cuda.synchronize()
    assert guess.shape[0] == B
classes = [(31, 11, 1), (61, 21, 2), (9, 4, 1)]
probs = [ql.build_problem(N=N, k_trans=kt, init_mode=im) for N, kt, im in classes]
ev = ql.RaggedEvaluator(probs)
class_of = rng.integers(0, len(classes), size=25)
Zf = ev.pack(class_of, [ql.initial_guess(probs[c]) + 1e-2 * rng.standard_normal(probs[c].n_nlp) for c in class_of])
Zd = torch.from_numpy(Zf).cuda()
off = ev.offsets(class_of)
zeros = lambda: {"f": torch.zeros(len(class_of), dtype=torch.float64, device="cuda"),
                 "grad": torch.zeros(int(off["z_off"][-1]), dtype=torch.float64, device="cuda"),
                 "g": torch.zeros(int(off["g_off"][-1]), dtype=torch.float64, device="cuda"),
                 "jac": torch.zeros(int(off["j_off"][-1]), dtype=torch.float64, device="cuda")}
a = ev.eval(class_of, Zd, out=zeros())           # (pre-zeroed: the padding element between rows is never written)
b = {"Z": Zd, **zeros()}                         # one qlnlp_eval_ragged_device launch per class
doff = {k: torch.from_numpy(v).cuda() for k, v in off.items()}
for c, nlp in enumerate(ev.nlps):
    nlp.eval_ragged(torch.from_numpy(np.nonzero(class_of == c)[0]).cuda(), b, doff, z_padded=True)
torch.cuda.synchronize()
for kname in ("f", "grad", "g", "jac"):
    assert torch.equal(a[kname], b[kname]), kname
print("sanitize case ok")
