"""Loops that let the library allocate every output (no ``out=``), the way a solver that keeps only the latest iterate
calls it: ``eval_batch`` at B = 4,096 (1.17 GB of outputs per call) and a small-B Hessian-vector product.  Host wall
time over the loop, closed by a device synchronise, so that both the launches and whatever the allocator does between
them are counted.  Prints the card and one line per loop.

    python tools/output_alloc_bench.py [--iters 200] [--rounds 3]
"""
from __future__ import annotations

import argparse
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()

    import numpy as np
    import torch
    import quadruped_landing_b200 as ql

    q = "name,power.limit,clocks.sm,clocks.max.sm"
    print("card:", subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                                  capture_output=True, text=True).stdout.strip(), flush=True)
    p = ql.default_problem()
    nlp = ql.HybridNLP.from_problem(p, hessian=True, products=True)
    rng = np.random.default_rng(0)

    def batch(B):
        Z = ql.initial_guess(p)[None, :] + 1e-2 * rng.standard_normal((B, p.n_nlp))
        Z[:, 19::20] = np.clip(Z[:, 19::20], 1e-3, 2e-2)
        return torch.from_numpy(Z).cuda()

    Zb = batch(4096)
    loops = {"eval_batch B=4096": lambda: nlp.eval_batch(Zb)}
    for B in (1, 64):
        Z = batch(B)
        mu = torch.from_numpy(rng.standard_normal((B, nlp.m_nlp))).cuda()
        V = torch.from_numpy(rng.standard_normal((B, nlp.n_nlp))).cuda()
        loops[f"hessian product B={B}"] = lambda Z=Z, mu=mu, V=V: nlp.eval_hessian_product_batch(Z, mu, V)

    for name, fn in loops.items():
        for _ in range(5):                                   # warm-up: modules, pools
            r = fn()
        del r
        torch.cuda.synchronize()
        ms = []
        for _ in range(args.rounds):
            t0 = time.perf_counter()
            for _ in range(args.iters):
                r = fn()                                     # the previous result is dropped here
            del r
            torch.cuda.synchronize()
            ms.append((time.perf_counter() - t0) * 1e3 / args.iters)
        print(f"{name:24s} ms/call median {statistics.median(ms):.4f} min {min(ms):.4f} max {max(ms):.4f}", flush=True)


if __name__ == "__main__":
    main()
