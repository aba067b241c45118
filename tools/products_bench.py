"""Throughput of the matrix-free products (eval_prod_kernel, hess_prod_kernel) at the default instance on one GPU, next
to what a caller does without them: materialise the Jacobian (eval_batch, SPARSE_TRUE and SPARSE_BLOCK) or the Hessian
(eval_hessian_batch) and multiply with a torch gather / index_add_.  Both routes run in the same process, alternating.

Per row: kernel time (CUDA events over many launches after a warm-up), evaluations/s, the algorithmic bytes per
evaluation (inputs read once, outputs written once), the achieved TB/s and its share of the device-to-device copy rate
measured in the same run.  Before timing, the timed outputs are checked bit for bit against a left fold of the
materialised values (the order include/qlnlp.h states).  Prints the card's name and power limit.

Usage:  python tools/products_bench.py [--reps 5] [--iters 20] [--out FILE]
"""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import quadruped_landing_b200 as ql


def fold(rows, cols, vals, vec, nout, transpose=False):
    """Left fold of vals * vec per output entry: rows over ascending columns, or (transpose) columns over ascending rows."""
    o, i = (cols - 1, rows - 1) if transpose else (rows - 1, cols - 1)
    acc = [None] * nout
    for e in np.lexsort((i, o)).tolist():
        t = float(vals[e]) * float(vec[i[e]])
        acc[o[e]] = t if acc[o[e]] is None else acc[o[e]] + t
    return np.array([np.nan if a is None else a for a in acc])


def timed(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e-3          # seconds per call


def copy_peak(iters):
    a = torch.empty(2 << 27, dtype=torch.float64, device="cuda")          # 2 GiB, well beyond L2
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    torch.cuda.synchronize()
    return 2 * a.numel() * 8 / timed(lambda: b.copy_(a), iters)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5, help="alternating repetitions of every route")
    ap.add_argument("--iters", type=int, default=20, help="launches per timed window")
    ap.add_argument("--out", help="also write the report to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to measure")
    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    say(f"card: {smi.stdout.strip() or smi.stderr.strip()}")
    p = ql.default_problem()
    nlp = ql.HybridNLP.from_problem(p, pattern="true", hessian=True, products=True)
    blk = ql.HybridNLP.from_problem(p, pattern="block")
    n, m = nlp.n_nlp, nlp.m_nlp
    peak = copy_peak(args.iters)
    say(f"measured device-to-device copy: {peak / 1e12:.2f} TB/s (2 GiB torch copy_, read + write)")
    rt, ct = (torch.from_numpy(a - 1).cuda() for a in nlp.jacobian_structure_arrays())
    rb, cb = (torch.from_numpy(a - 1).cuda() for a in blk.jacobian_structure_arrays())
    hr, hc = nlp.hessian_structure_arrays()
    off = hr != hc
    mr = torch.from_numpy(np.concatenate([hr, hc[off]]) - 1).cuda()
    mc = torch.from_numpy(np.concatenate([hc, hr[off]]) - 1).cuda()
    hidx = torch.from_numpy(np.concatenate([np.arange(len(hr)), np.nonzero(off)[0]])).cuda()
    rng = np.random.default_rng(0)
    base = ql.initial_guess(p)
    B0 = 4096
    Z0 = base[None, :] + 1e-2 * rng.standard_normal((B0, n))
    Z0[:, 19::20] = np.clip(Z0[:, 19::20], 1e-3, 2e-2)
    bytes_per = {"Jw": 8 * (2 * n + m), "J'y": 8 * (2 * n + m), "Jw + J'y + g": 8 * (3 * n + 3 * m),
                 "Hv": 8 * (3 * n + m)}
    say(f"default instance: n_nlp {n}, m_nlp {m}; algorithmic bytes per evaluation: "
        + ", ".join(f"{k} {v:,}" for k, v in bytes_per.items()))
    for B in (4096, 65536):
        ev = lambda d: torch.zeros((B, d + 1), dtype=torch.float64, device="cuda")[:, :d]
        Z = ev(n)
        Z.copy_(torch.from_numpy(Z0).cuda().repeat(B // B0, 1))
        w, v = ev(n), ev(n)
        y, lam = ev(m), ev(m)
        for t in (w, v, y, lam):
            t.normal_()
        o_jw, o_jty, o_both, o_hv = {}, {}, {}, ev(n)
        gbuf = {}
        mat = {"true": {}, "block": {}}
        hbuf = {}
        routes = {
            "Jw": lambda: nlp.eval_products_batch(Z, w=w, out=o_jw),
            "J'y": lambda: nlp.eval_products_batch(Z, y=y, out=o_jty),
            "Jw + J'y + g": lambda: nlp.eval_products_batch(Z, w=w, y=y, want=("g",), out=o_both),
            "Hv": lambda: nlp.eval_hessian_product_batch(Z, lam, v, out=o_hv),
        }

        def mm_jw(h, r, c, buf):
            vals = h.eval_batch(Z, want=("jac",), out=buf)["jac"]
            return torch.zeros((B, m), dtype=torch.float64, device="cuda").index_add_(1, r, vals * w[:, c])

        def mm_jty(h, r, c, buf):
            vals = h.eval_batch(Z, want=("jac",), out=buf)["jac"]
            return torch.zeros((B, n), dtype=torch.float64, device="cuda").index_add_(1, c, vals * y[:, r])

        def mm_both(h, r, c, buf):
            vals = h.eval_batch(Z, want=("g", "jac"), out=buf)["jac"]
            a = torch.zeros((B, m), dtype=torch.float64, device="cuda").index_add_(1, r, vals * w[:, c])
            return a, torch.zeros((B, n), dtype=torch.float64, device="cuda").index_add_(1, c, vals * y[:, r])

        def mm_hv():
            H = nlp.eval_hessian_batch(Z, lam, out=hbuf.get("H"))
            hbuf["H"] = H
            return torch.zeros((B, n), dtype=torch.float64, device="cuda").index_add_(1, mr, H[:, hidx] * v[:, mc])

        base_routes = {
            "Jw": {"true": lambda: mm_jw(nlp, rt, ct, mat["true"]), "block": lambda: mm_jw(blk, rb, cb, mat["block"])},
            "J'y": {"true": lambda: mm_jty(nlp, rt, ct, mat["true"]), "block": lambda: mm_jty(blk, rb, cb, mat["block"])},
            "Jw + J'y + g": {"true": lambda: mm_both(nlp, rt, ct, mat["true"]), "block": lambda: mm_both(blk, rb, cb, mat["block"])},
            "Hv": {"true": mm_hv},
        }
        # bit-for-bit check of the timed outputs against the fold of the materialised values (two rows)
        for fn in routes.values():
            fn()
        vals = nlp.eval_batch(Z, want=("jac",))["jac"]
        Hm = nlp.eval_hessian_batch(Z, lam)
        torch.cuda.synchronize()
        rows, cols = nlp.jacobian_structure_arrays()
        mrn, mcn = mr.cpu().numpy() + 1, mc.cpu().numpy() + 1
        for b in (0, B - 1):
            V, Hb = vals[b].cpu().numpy(), Hm[b].cpu().numpy()[hidx.cpu().numpy()]
            fw = fold(rows, cols, V, w[b].cpu().numpy(), m)
            fy = fold(rows, cols, V, y[b].cpu().numpy(), n, transpose=True)
            fh = fold(mrn, mcn, Hb, v[b].cpu().numpy(), n)
            assert np.array_equal(o_jw["jw"][b].cpu().numpy(), fw) and np.array_equal(o_both["jw"][b].cpu().numpy(), fw)
            assert np.array_equal(o_jty["jty"][b].cpu().numpy(), fy) and np.array_equal(o_both["jty"][b].cpu().numpy(), fy)
            assert np.array_equal(o_hv[b].cpu().numpy(), fh)
        say(f"B = {B}: outputs equal the fold of the materialised matrices bit for bit (rows 0 and {B - 1})")
        # warm-up of every timed shape, then alternating repetitions
        for fn in list(routes.values()) + [f for d in base_routes.values() for f in d.values()]:
            for _ in range(3):
                fn()
        torch.cuda.synchronize()
        t = {}
        for _ in range(args.reps):
            for name, fn in routes.items():
                t.setdefault((name, "product"), []).append(timed(fn, args.iters))
                for pat, bf in base_routes[name].items():
                    t.setdefault((name, f"materialise {pat} + torch"), []).append(timed(bf, max(2, args.iters // 4)))
        say(f"{'B':>6} {'product':<14} {'route':<30} {'time/launch':>12} {'spread':>8} {'evals/s':>10} {'TB/s':>6} {'of copy':>8}")
        for (name, route), ts in t.items():
            s = float(np.median(ts))
            bw = bytes_per[name] * B / s
            say(f"{B:>6} {name:<14} {route:<30} {s * 1e3:>9.4f} ms {100 * (max(ts) - min(ts)) / s:>6.1f} % "
                f"{B / s / 1e6:>7.1f} M {bw / 1e12:>6.2f} {100 * bw / peak:>6.1f} %")
        del mat["true"], mat["block"], hbuf
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
