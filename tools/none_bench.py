import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import quadruped_landing_b200 as ql
p = ql.default_problem(); nlp = ql.HybridNLP.from_problem(p)
rng = np.random.default_rng(0)
Z = ql.initial_guess(p)[None, :] + 1e-2 * rng.standard_normal((4096, p.n_nlp))
for Bt in (4096, 65536):
    Zt = torch.zeros((Bt, 1216), dtype=torch.float64, device="cuda")[:, :1215]
    Zt.copy_(torch.from_numpy(Z).cuda().repeat(Bt // 4096, 1))
    for want in (("f", "grad", "g"), ("g",), ("f",)):
        out = nlp.eval_batch(Zt, want=want)
        for _ in range(10): nlp.eval_batch(Zt, want=want, out=out)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n = 50 if Bt == 4096 else 10
        e0.record()
        for _ in range(n): nlp.eval_batch(Zt, want=want, out=out)
        e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        print(f"B={Bt} {'+'.join(want):10s} {Bt / ms * 1e3 / 1e6:8.2f} M evals/s  {nlp.launch_info()['blocks_per_sm']} warps/SM")
