"""Replay time of a CUDA graph that holds every launcher (the graph of
tests/test_gpu_parity.py::test_every_launcher_can_be_captured_in_a_cuda_graph): the products, the Hessian, the Hessian
products, the KKT solve and a kinematic handle's evaluation at B = 600 on the default problem.

    python tools/graph_replay_bench.py [--replays 200] [--repeats 5]

Prints one JSON line: the median and spread of the per-replay time (CUDA events around `replays` back-to-back replays,
`repeats` times), the eager time of the same launches, and the card.  QLNLP_LIB selects another build of the library
(tools/ab_bench.py), so two builds are compared by running this once with each.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--replays", type=int, default=200)
    ap.add_argument("--repeats", type=int, default=5)
    a = ap.parse_args()
    import torch
    import quadruped_landing_b200 as ql
    from conftest import perturbed_batch

    p = ql.default_problem()
    nlp = ql.HybridNLP.from_problem(p, pattern="true", hessian=True)
    kin = ql.HybridNLP.from_problem(p, kinematics=True)
    B, n, m = 600, nlp.n_nlp, nlp.m_nlp
    rng = np.random.default_rng(12)
    cuda = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    Z = cuda(perturbed_batch(p, [ql.initial_guess(p)], B, 1e-2, 12))
    lam, sigma = cuda(1e-4 * rng.standard_normal((B, m))), cuda(np.full(B, 1e-4))
    w, y, V = cuda(rng.standard_normal((B, n))), cuda(rng.standard_normal((B, m))), cuda(rng.standard_normal((B, n)))
    dc, sx = cuda(rng.uniform(1e-2, 1.0, (B, m))), cuda(rng.uniform(1.0, 10.0, (B, n)))
    r1, r2 = cuda(rng.standard_normal((B, n))), cuda(rng.standard_normal((B, m)))
    jac = nlp.eval_batch(Z, want=("jac",))["jac"]
    out = {"prod": nlp.eval_products_batch(Z, w=w, y=y, want=("f", "g")), "hess": nlp.eval_hessian_batch(Z, lam, sigma=sigma),
           "hv": nlp.eval_hessian_product_batch(Z, lam, V, sigma=sigma), "kin": kin.eval_batch(Z)}
    out["kkt"] = nlp.kkt_solve_batch(out["hess"], jac, dc, r1, r2, sx=sx)

    def run():
        nlp.eval_products_batch(Z, w=w, y=y, want=("f", "g"), out=out["prod"])
        nlp.eval_hessian_batch(Z, lam, sigma=sigma, out=out["hess"])
        nlp.eval_hessian_product_batch(Z, lam, V, sigma=sigma, out=out["hv"])
        nlp.kkt_solve_batch(out["hess"], jac, dc, r1, r2, sx=sx, out=out["kkt"])
        kin.eval_batch(Z, out=out["kin"])

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        run()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        run()
    torch.cuda.synchronize()

    def timed(fn):
        for _ in range(10):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(a.repeats):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.replays):
                fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3 / a.replays)
        return ts

    rep = timed(g.replay)
    eager = timed(run)
    print(json.dumps({"lib": os.environ.get("QLNLP_LIB", "default"), "B": B, "replays": a.replays,
                      "replay_us_median": float(np.median(rep)), "replay_us_min": min(rep), "replay_us_max": max(rep),
                      "eager_us_median": float(np.median(eager)), "card": card()}))


if __name__ == "__main__":
    main()
