"""Does compressible device memory speed up the evaluator's output stream on this GPU?

Times the headline launch (C2 inputs, f + grad + g + SPARSE_BLOCK Jacobian, ``ql::eval_kernel<1, 1, 0>``) writing
into plain ``cudaMalloc``-style memory (``torch.empty``) against the same launch writing into a ``qlnlp_device_alloc``
block (``cuMemCreate`` with generic compression where the device offers it).  The two arms alternate, round after
round, so that clock and neighbour drift hit both alike.  A device-to-device ``cudaMemcpyAsync`` of the same bytes (an
image of real Jacobian rows, then random doubles) into each kind of memory separates what the allocation does from what
the kernel does.  Prints the card, its power limit and SM clock, then one line per measurement.

    python tools/compress_probe.py [--rounds 7] [--launches 500] [--big-launches 200]
"""
from __future__ import annotations

import argparse
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
    try:
        return subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                   # noqa: BLE001
        return f"nvidia-smi unavailable: {e}"


def timed(torch, fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        fn(i)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / n


def plain_outputs(torch, nlp, B):
    from quadruped_landing_b200.evaluator import even_ld
    dev = torch.device("cuda", nlp.device)
    out = {"f": torch.empty(B, dtype=torch.float64, device=dev)}
    for k, w in (("grad", nlp.n_nlp), ("g", nlp.m_nlp), ("jac", nlp.nnz_batch)):
        out[k] = torch.empty((B, even_ld(w)), dtype=torch.float64, device=dev)[:, :w]
    return out


def spread(xs):
    return f"median {statistics.median(xs):.4f} min {min(xs):.4f} max {max(xs):.4f}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--launches", type=int, default=500, help="launches per round at B = 4,096")
    ap.add_argument("--big-launches", type=int, default=200, help="launches per round at B = 65,536")
    args = ap.parse_args()

    import numpy as np
    import torch
    import bench
    import quadruped_landing_b200 as ql
    from quadruped_landing_b200.evaluator import device_alloc_info

    print("card:", card(), flush=True)
    prob = ql.default_problem()
    nlp = ql.HybridNLP.from_problem(prob, device=0)
    dev = torch.device("cuda", 0)
    host_sets = bench.make_inputs(prob, 0, bench.N_INPUT_SETS)
    want = ("f", "grad", "g", "jac")

    for B, n in ((4096, args.launches), (65536, args.big_launches)):
        rep = B // bench.B_PER_GPU
        Zs = [bench.padded(torch, np.tile(z, (rep, 1)), dev) for z in host_sets]
        arms = {"plain": plain_outputs(torch, nlp, B), "comp": nlp.alloc_outputs(B, want)}
        print(f"B={B} comp block: {device_alloc_info(arms['comp']['jac'])}", flush=True)
        for a in arms.values():                                  # warm-up and first touch
            for i in range(20):
                nlp.eval_batch(Zs[i % len(Zs)], want=want, out=a)
        torch.cuda.synchronize()
        same = all(torch.equal(arms["plain"][k], arms["comp"][k]) for k in want)
        print(f"B={B} outputs bit-identical between arms: {same}", flush=True)
        ms = {k: [] for k in arms}
        for r in range(args.rounds):
            order = ("plain", "comp") if r % 2 == 0 else ("comp", "plain")
            for k in order:
                ms[k].append(timed(torch, lambda i: nlp.eval_batch(Zs[i % len(Zs)], want=want, out=arms[k]), n))
        for k in arms:
            rates = [B / (m * 1e-3) / 1e6 for m in ms[k]]
            gbs = [B * bench.BYTES_FULL / (m * 1e-3) / 1e12 for m in ms[k]]
            print(f"B={B} kernel {k:5s}: ms/launch {spread(ms[k])} | M evals/s {spread(rates)} | "
                  f"algorithmic TB/s {spread(gbs)}", flush=True)

        if B == 4096:
            # copies of the Jacobian buffer's bytes into each kind of memory
            full = lambda t: t.as_strided((t.shape[0], t.stride(0)), (t.stride(0), 1))   # padded rows: one memcpy
            src_rows = full(arms["plain"]["jac"]).clone()          # real rows, plain memory
            src_rand = torch.rand_like(src_rows)
            dst = {k: full(a["jac"]) for k, a in arms.items()}
            nbytes = src_rows.numel() * 8
            for label, src in (("real-rows image", src_rows), ("random doubles", src_rand)):
                cm = {k: [] for k in dst}
                for r in range(args.rounds):
                    order = ("plain", "comp") if r % 2 == 0 else ("comp", "plain")
                    for k in order:
                        cm[k].append(timed(torch, lambda i: dst[k].copy_(src), 50))
                for k in dst:
                    tbs = [2 * nbytes / (m * 1e-3) / 1e12 for m in cm[k]]
                    print(f"B={B} memcpy {label:15s} -> {k:5s}: ms {spread(cm[k])} | read+write TB/s {spread(tbs)}",
                          flush=True)
        del arms, Zs
        torch.cuda.synchronize()
    print("card after:", card(), flush=True)


if __name__ == "__main__":
    main()
