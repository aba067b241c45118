"""Throughput of the batched KKT solve (kkt_kernel) at the default instance (N = 61, k_trans = 21) on one GPU, next to
a CPU baseline in the same process: scipy factorising the same problems one by one (splu of the assembled sparse KKT
matrix) on all host cores, over a sample.  Then the factor / solve split in the same process: kkt_factor_kernel alone,
kkt_solve_factored_kernel with one right-hand side per factor (R = B) and with four per factor through `index`
(R = 4B), each launch alternating with a one-shot solve, and one factorisation plus two factored solves against two
one-shot solves.  The cost of one refinement step of kkt_solve_refined_batch: kkt_residual_kernel alone, and residual +
factored solve + the two device adds (px += dpx, pl += dpl) as one timed call.

Inputs: C3-style decision vectors (device-built guesses of the drop-height x pitch sweep, perturbed), seeded
multipliers (scale 1e-4), objective factor 1e-4 (at 1 the objective's x-h second derivatives make these M
indefinite), Hessians and SPARSE_TRUE Jacobians from the device kernels, seeded dc in [1e-2, 1], sx in [1, 10], r1, r2.
Timing: CUDA events over many launches after a warm-up.  Bytes and flops come from the counts below (per problem).
Prints the card's name and power limit; the sampled GPU steps are checked against the CPU solves.

Usage:  python tools/kkt_bench.py [--iters 20] [--sample 512] [--out FILE]
"""
import argparse
import os
import subprocess
import sys
import time
from concurrent.futures import ProcessPoolExecutor

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla
import torch

import quadruped_landing_b200 as ql

HBM_TBS = 7.7          # HGX B200 data sheet, one GPU
FP64_TFLOPS = 37.0     # profiles/r01_fp64_peak.log: DFMA throughput measured on one B200


def stream_bytes(nlp):
    """Input and output streams: W, J, sx, dc, r1, r2 read once, px, pl written once."""
    n, m = nlp.n_nlp, nlp.m_nlp
    return 8 * (nlp.nnz_hess + nlp.nnz + n + m + n + m + n + m)


def scratch_bytes(N):
    """Factor scratch: L_kk packed (210, 120 at knot N) and y_k (20, 15 at knot N), written once and read once."""
    return 2 * 8 * ((N - 1) * (210 + 20) + (120 + 15))


def kernel_flops(N):
    """Floating-point operations the kernel executes per problem (multiply-adds count 2, structural zeros of the dense
    34 x 20 local Jacobian included), from the loops of qlnlp_kkt.cuh."""
    S = 34
    total = 0
    for k in range(1, N + 1):
        nk = 20 if k < N else 15
        T = nk * (nk + 1) // 2
        f = T * (1 + 3 * S) + nk + nk * (S * 3 + 1)                  # M_kk and b_k from G, W, sx, r1, r2
        if k > 1:
            f += 15 * 20 + 120 * (2 * 20 + 1) + 15 * (2 * 20 + 1)     # apply E, rank-15 update of M_kk and b_k
        f += sum(1 + (nk - 1 - j) + sum(2 * (i - j) for i in range(j + 1, nk)) for j in range(nk))   # Cholesky
        f += sum(1 + 2 * (nk - 1 - j) for j in range(nk))             # y_k = L^-1 b
        if k < N:
            f += 15 * sum(1 + 2 * j + 1 for j in range(20))           # X_k = D^-1 A_k L^-T
            f += 20 * 15 * 4 + sum(1 + 2 * (19 - j) for j in range(20)) + 20     # backward: L^-1 (A' D^-1 E x)
        f += sum(1 + 2 * j for j in range(nk))                        # x_k = L^-T r
        f += S * (2 * nk + 4) + S * 2                                 # pl rows; 1/dc, r2/dc per slot
        total += f
    return total


def _knot_flops(N, k):
    """Operations of knot k by step, from the loops of qlnlp_kkt.cuh (see kernel_flops)."""
    S = 34
    nk = 20 if k < N else 15
    T = nk * (nk + 1) // 2
    return {
        "mkk": T * (1 + 3 * S) + (15 * 20 + 120 * (2 * 20 + 1) if k > 1 else 0),         # M_kk, E, rank-15 update
        "chol": sum(1 + (nk - 1 - j) + sum(2 * (i - j) for i in range(j + 1, nk)) for j in range(nk)),
        "xk": 15 * sum(1 + 2 * j + 1 for j in range(20)) if k < N else 0,                  # X_k = D^-1 A_k L^-T
        "bk": nk + nk * (S * 3 + 1) + (15 * (2 * 20 + 1) if k > 1 else 0),                 # b_k - X_(k-1) y_(k-1)
        "yk": sum(1 + 2 * (nk - 1 - j) for j in range(nk)),                                # y_k = L^-1 b
        "back": (20 * 15 * 4 + sum(1 + 2 * (19 - j) for j in range(20)) + 20 if k < N else 0)
                + sum(1 + 2 * j for j in range(nk)) + S * (2 * nk + 4),                    # x_k and the pl rows
        "rdc": S,                                                                          # 1/dc per slot, one gather
    }


def factor_flops(N):
    """kkt_factor_kernel per problem: M_kk, Cholesky and X_k of every knot."""
    return sum(t["mkk"] + t["chol"] + t["xk"] + t["rdc"] for t in (_knot_flops(N, k) for k in range(1, N + 1)))


def solve_flops(N):
    """kkt_solve_factored_kernel per right-hand side: b_k, y_k, the backward sweep (1/dc in both sweeps' gathers)."""
    return sum(t["bk"] + t["yk"] + t["back"] + 2 * t["rdc"] for t in (_knot_flops(N, k) for k in range(1, N + 1)))


def factor_bytes(nlp):
    """kkt_factor_kernel per problem: W, J, sx, dc read once, the factor row written once."""
    n, m = nlp.n_nlp, nlp.m_nlp
    return 8 * (nlp.nnz_hess + nlp.nnz + n + m) + 8 * nlp.kkt_factor_size


def solve_bytes(nlp):
    """kkt_solve_factored_kernel per right-hand side: the factor row read once (the backward sweep's second read of
    L_kk, J and dc not counted), r1, r2 read, y_k written to px and read back, px and pl written."""
    n, m = nlp.n_nlp, nlp.m_nlp
    return 8 * nlp.kkt_factor_size + 8 * (n + m) + 16 * n + 8 * (n + m)


def residual_flops(N, m):
    """kkt_residual_kernel per problem: one fused multiply-add per term of every entry (2 flops), the knot-local
    structural zeros included: s1 folds its knot's W row and 34 slots, s2 at most 20 columns + the -I + dc."""
    return sum(2 * nk * (nk + 34 + 1) for nk in [20] * (N - 1) + [15]) + 2 * m * 22


def residual_bytes(nlp):
    """kkt_residual_kernel per problem: W, J, sx, dc, r1, r2, px, pl read once, s1, s2 written once."""
    n, m = nlp.n_nlp, nlp.m_nlp
    return 8 * (nlp.nnz_hess + nlp.nnz + n + m) + 8 * 3 * (n + m)


def _cpu_solve(args):
    hs, hv, js, jv, sx, dc, r1, r2 = args
    n, m = len(sx), len(dc)
    hr, hc = hs[0] - 1, hs[1] - 1
    off = hr != hc
    W = sp.coo_matrix((np.concatenate([hv, hv[off]]), (np.concatenate([hr, hc[off]]), np.concatenate([hc, hr[off]]))),
                      shape=(n, n))
    J = sp.coo_matrix((jv, (js[0] - 1, js[1] - 1)), shape=(m, n))
    K = sp.bmat([[W + sp.diags(sx), J.T], [J, -sp.diags(dc)]], format="csc")
    z = spla.splu(K).solve(np.concatenate([r1, r2]))
    return z


def _cpu_batch(chunk):
    return [_cpu_solve(a) for a in chunk]


def split(a, log, nlp, B, hess, jac, dc, sx, r1, r2, out, gen):
    """The factor / solve split at batch B, each new launch alternating with a one-shot solve in one stream."""
    n, m = nlp.n_nlp, nlp.m_nlp
    R4 = 4 * B
    q1 = torch.randn((R4, n), generator=gen, device="cuda", dtype=torch.float64)
    q2 = torch.randn((R4, m), generator=gen, device="cuda", dtype=torch.float64)
    index = torch.arange(B, dtype=torch.int64, device="cuda").repeat_interleave(4)
    fac = nlp.kkt_factor_batch(hess, jac, dc, sx=sx)
    one = nlp.kkt_solve_factored_batch(fac[0], r1, r2)
    four = nlp.kkt_solve_factored_batch(fac[0], q1, q2, index=index)
    res = nlp.kkt_residual_batch(hess, jac, dc, one[0], one[1], r1, r2, sx=sx)
    cor = nlp.kkt_solve_factored_batch(fac[0], res[0], res[1])
    px, pl = one[0].clone(), one[1].clone()
    torch.cuda.synchronize()
    same = all(torch.equal(x, y) for x, y in zip(one, out))

    def refine_step():
        nlp.kkt_residual_batch(hess, jac, dc, px, pl, r1, r2, sx=sx, out=res)
        nlp.kkt_solve_factored_batch(fac[0], res[0], res[1], out=cor)
        px.add_(cor[0])
        pl.add_(cor[1])

    calls = {
        "one-shot": lambda: nlp.kkt_solve_batch(hess, jac, dc, r1, r2, sx=sx, out=out),
        "factor": lambda: nlp.kkt_factor_batch(hess, jac, dc, sx=sx, out=fac),
        "solve R=B": lambda: nlp.kkt_solve_factored_batch(fac[0], r1, r2, out=one),
        "solve R=4B": lambda: nlp.kkt_solve_factored_batch(fac[0], q1, q2, index=index, out=four),
        "residual": lambda: nlp.kkt_residual_batch(hess, jac, dc, one[0], one[1], r1, r2, sx=sx, out=res),
        "refine step": refine_step,
    }
    for f in calls.values():
        f()
    torch.cuda.synchronize()
    ev = {k: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.iters)]
          for k in calls}
    for i in range(a.iters):
        for k, f in calls.items():
            e0, e1 = ev[k][i]
            e0.record()
            f()
            e1.record()
    torch.cuda.synchronize()
    med = {}
    for k in calls:
        ms = sorted(e0.elapsed_time(e1) for e0, e1 in ev[k])
        med[k] = ms[len(ms) // 2]
        rows = R4 if k == "solve R=4B" else B
        per = {"one-shot": (stream_bytes(nlp) + scratch_bytes(nlp.N), kernel_flops(nlp.N)),
               "factor": (factor_bytes(nlp), factor_flops(nlp.N)),
               "residual": (residual_bytes(nlp), residual_flops(nlp.N, nlp.m_nlp)),
               "refine step": (residual_bytes(nlp) + solve_bytes(nlp) + 8 * 3 * (nlp.n_nlp + nlp.m_nlp),
                               residual_flops(nlp.N, nlp.m_nlp) + solve_flops(nlp.N))}.get(
                   k, (solve_bytes(nlp), solve_flops(nlp.N)))
        rate = rows / (med[k] * 1e-3)
        bw, fr = per[0] * rate / 1e12, per[1] * rate / 1e12
        log(f"  B={B} {k:>10}: {med[k]:.3f} ms median (min {ms[0]:.3f}, max {ms[-1]:.3f}) over {a.iters} alternating "
            f"launches; {rate / 1e6:.3f} M rows/s; {bw:.3f} TB/s ({100 * bw / HBM_TBS:.1f} % of HBM), {fr:.3f} TFLOP/s "
            f"({100 * fr / FP64_TFLOPS:.1f} % of DFMA)")
    st = [t.cpu().numpy() for t in (fac[1], one[2], four[2])]
    log(f"  B={B}: factored solve R=B equals the one-shot bits: {same}; status 0: factor {int((st[0] == 0).sum())}, "
        f"R=B {int((st[1] == 0).sum())} of {B}, R=4B {int((st[2] == 0).sum())} of {R4}")
    two = 2 * med["one-shot"]
    split_ms = med["factor"] + 2 * med["solve R=B"]
    log(f"  B={B}: factor + 2 factored solves {split_ms:.3f} ms vs 2 one-shot solves {two:.3f} ms "
        f"({'faster' if split_ms < two else 'NOT faster'}: {two / split_ms:.2f}x); a factored solve costs "
        f"{med['solve R=B'] / med['one-shot']:.3f} of a one-shot solve, the factor {med['factor'] / med['one-shot']:.3f}")
    log(f"  B={B}: one refinement step (residual + factored solve + 2 adds) {med['refine step']:.3f} ms = "
        f"{med['refine step'] / med['one-shot']:.3f} of a one-shot solve; the residual alone {med['residual']:.3f} ms; "
        f"3-step refined solve ~ factor + {1 + 3} factored solves + 3 residuals = "
        f"{med['factor'] + med['solve R=B'] + 3 * med['refine step']:.3f} ms")
    del fac, one, four, q1, q2, res, cor, px, pl


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--sample", type=int, default=512)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lines = []

    def log(s=""):
        print(s, flush=True)
        lines.append(s)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True)
    log(f"card: {torch.cuda.get_device_name(0)}; nvidia-smi name, power.limit: {smi.stdout.strip().splitlines()[0]}")
    p = ql.default_problem()
    nlp = ql.HybridNLP.from_problem(p, pattern="true", hessian=True)
    N = p.N
    sb, fb, fl = stream_bytes(nlp), scratch_bytes(N), kernel_flops(N)
    log(f"instance N={N} k_trans={p.k_trans}: n_nlp={nlp.n_nlp} m_nlp={nlp.m_nlp} nnz_true={nlp.nnz} "
        f"nnz_hess={nlp.nnz_hess}")
    log(f"per problem: streams {sb:,} B, factor scratch {fb:,} B (write + read), kernel flops {fl:,} "
        f"({fl / N:,.0f} per knot)")
    log(f"factor row {nlp.kkt_factor_size:,} doubles ({8 * nlp.kkt_factor_size:,} B); factor: {factor_bytes(nlp):,} B, "
        f"{factor_flops(N):,} flops per problem; factored solve: {solve_bytes(nlp):,} B, {solve_flops(N):,} flops per "
        f"right-hand side")
    log(f"host cores: {os.cpu_count()}")
    gen = torch.Generator(device="cuda").manual_seed(0)
    for B in (4096, 65536):
        side = int(round(B ** 0.5))
        x0 = ql.sweep_initial_states(p.model, np.linspace(0.25, 3.0, side), np.linspace(-40.0, -5.0, B // side))
        x0d = torch.from_numpy(x0).cuda()
        Z = nlp.initial_guess_batch(x0d)
        Z.add_(1e-3 * torch.randn(Z.shape, generator=gen, device="cuda", dtype=torch.float64))
        rnd = lambda w: torch.rand((B, w), generator=gen, device="cuda", dtype=torch.float64)
        lam = 1e-4 * torch.randn((B, nlp.m_nlp), generator=gen, device="cuda", dtype=torch.float64)
        jac = nlp.eval_batch(Z, x0=x0d, want=("jac",))["jac"]
        hess = nlp.eval_hessian_batch(Z, lam, sigma=torch.full((B,), 1e-4, dtype=torch.float64, device="cuda"))
        dc, sx = 1e-2 + 0.99 * rnd(nlp.m_nlp), 1.0 + 9.0 * rnd(nlp.n_nlp)
        r1 = torch.randn((B, nlp.n_nlp), generator=gen, device="cuda", dtype=torch.float64)
        r2 = torch.randn((B, nlp.m_nlp), generator=gen, device="cuda", dtype=torch.float64)
        out = nlp.kkt_solve_batch(hess, jac, dc, r1, r2, sx=sx)
        for _ in range(3):
            nlp.kkt_solve_batch(hess, jac, dc, r1, r2, sx=sx, out=out)
        torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.iters)]
        for e0, e1 in ev:
            e0.record()
            nlp.kkt_solve_batch(hess, jac, dc, r1, r2, sx=sx, out=out)
            e1.record()
        torch.cuda.synchronize()
        ms = sorted(e0.elapsed_time(e1) for e0, e1 in ev)
        med = ms[len(ms) // 2]
        rate = B / (med * 1e-3)
        st = out[2].cpu().numpy()
        log(f"B={B}: kernel {med:.3f} ms median (min {ms[0]:.3f}, max {ms[-1]:.3f}) over {a.iters} launches; "
            f"{rate / 1e6:.3f} M solves/s; status 0 for {int((st == 0).sum())} of {B}")
        bw = (sb + fb) * rate / 1e12
        fr = fl * rate / 1e12
        log(f"  streams + scratch {bw:.3f} TB/s ({100 * bw / HBM_TBS:.1f} % of {HBM_TBS} TB/s HBM); streams alone "
            f"{sb * rate / 1e12:.3f} TB/s; {fr:.3f} TFLOP/s fp64 ({100 * fr / FP64_TFLOPS:.1f} % of {FP64_TFLOPS} "
            f"measured DFMA peak); closer bound: {'memory' if bw / HBM_TBS > fr / FP64_TFLOPS else 'fp64'}")
        if B == 4096:
            hs, js = nlp.hessian_structure_arrays(), nlp.jacobian_structure_arrays()
            idx = np.arange(0, B, max(1, B // a.sample))[:a.sample]
            cpu = lambda t: t[idx].cpu().numpy()
            H, Jv, SX, DC, R1, R2 = (cpu(t) for t in (hess, jac, sx, dc, r1, r2))
            args = [(hs, H[i], js, Jv[i], SX[i], DC[i], R1[i], R2[i]) for i in range(len(idx))]
            ncpu = os.cpu_count()
            chunks = [args[i::ncpu] for i in range(ncpu)]
            with ProcessPoolExecutor(ncpu) as pool:
                list(pool.map(_cpu_batch, [c[:1] for c in chunks]))          # warm the workers
                t0 = time.perf_counter()
                res = list(pool.map(_cpu_batch, chunks))
                t1 = time.perf_counter()
            cpu_rate = len(idx) / (t1 - t0)
            zc = np.empty((len(idx), nlp.n_nlp + nlp.m_nlp))
            for c, r in enumerate(res):
                zc[c::ncpu] = np.array(r)
            zg = np.concatenate([cpu(out[0]), cpu(out[1])], axis=1)
            rel = np.abs(zg - zc).max(axis=1) / np.abs(zc).max(axis=1)
            log(f"  CPU baseline (scipy splu, one problem at a time, {ncpu} processes, {len(idx)} problems): "
                f"{cpu_rate:,.0f} solves/s; GPU / CPU = {rate / cpu_rate:,.0f}x; max relative difference of the steps "
                f"{rel.max():.2e}")
        split(a, log, nlp, B, hess, jac, dc, sx, r1, r2, out, gen)
        del out, hess, jac, Z, lam, dc, sx, r1, r2
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
