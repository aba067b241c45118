import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import quadruped_landing_b200 as ql
from oracle.oracle import Oracle
for N, kt, im in [(257, 100, 1), (512, 2, 2), (1024, 1000, 1)]:
    p = ql.build_problem(N=N, k_trans=kt, init_mode=im)
    o = Oracle(p)
    rng = np.random.default_rng(N)
    Z = rng.normal(size=(40, p.n_nlp)); Z[:, 19::20] = rng.uniform(1e-3, 2e-2, size=(40, N - 1))
    for pattern in ("block", "true"):
        nlp = ql.HybridNLP.from_problem(p, pattern=pattern)
        out = nlp.eval_batch(torch.from_numpy(Z).cuda()); torch.cuda.synchronize()
        ref = o.eval_batch(Z, pattern=pattern)
        ok = all(np.all(np.abs(out[k].cpu().numpy() - ref[k]) <= 1e-14 + 1e-12 * np.abs(ref[k])) for k in ref)
        print(N, kt, im, pattern, "ok" if ok else "MISMATCH", nlp.launch_info())
