"""SURVEY.md 8d C4: 32,768 problems of 12 mixed classes in flat arrays; throughput of the ragged path."""
import sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import quadruped_landing_b200 as ql
classes = [(N, kt, im) for (N, kt) in [(31, 11), (41, 14), (61, 21), (81, 27), (101, 34), (121, 41)] for im in (1, 2)]
probs = [ql.build_problem(N=N, k_trans=kt, init_mode=im) for N, kt, im in classes]
ev = ql.RaggedEvaluator(probs)
rng = np.random.default_rng(7)
B = 32768
class_of = rng.integers(0, len(classes), size=B)
off = ev.offsets(class_of)
guesses = [ql.initial_guess(p) for p in probs]
Zf = ev.pack(class_of, [guesses[c] + 1e-2 * rng.standard_normal(probs[c].n_nlp) for c in class_of])
Zd = torch.from_numpy(Zf).cuda()
plan = ev.plan(class_of, Zd.device)
bytes_total = 8 * int(sum(2 * ev.n[c] + ev.m[c] + ev.nnz[c] + 1 for c in class_of))
out = ev.eval(plan, Zd); torch.cuda.synchronize()
for want in (("f", "grad", "g", "jac"), ("g", "jac")):
    for _ in range(2):
        ev.eval(plan, Zd, out=out, want=want)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 8
    e0.record()
    for _ in range(n):
        ev.eval(plan, Zd, out=out, want=want)
    e1.record(); torch.cuda.synchronize()
    dt = e0.elapsed_time(e1) / n * 1e-3
    print(f"C4 ragged ONE launch {'+'.join(want):12s}: B={B}, {bytes_total / 1e9:.2f} GB per pass, "
          f"{dt * 1e3:.2f} ms  {B / dt / 1e6:.2f} M evals/s  {bytes_total / dt / 1e12:.2f} TB/s  {ev.nlps[0].launch_info()}")
