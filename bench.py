#!/usr/bin/env python3
"""Benchmark of the hot path: batched NLP evaluations per second (f + grad + g + sparse Jacobian).

    python bench.py --gpus N --steps K --warmup W            # this framework (CUDA, sm_100a)
    python bench.py --impl reference --gpus N --steps K ...  # CPU restatement of the reference algorithm
    torchrun --nproc-per-node N bench.py --gpus N ...        # one rank per GPU

Headline (BASELINE.json configs[1], SURVEY.md 8d C2): a step = one fused launch over one batch of B=4096 perturbed
decision vectors of the reference's default landing NLP (N=61 knots, k_trans=21, init_mode=1) per GPU, producing f,
grad_f, g and the SPARSE_BLOCK Jacobian values (285,480 algorithmic bytes per evaluation).  `e2e` is the same batch
through the C ABI on HOST buffers (qlnlp_eval_batch_host), copies inside the timed region.
Extra keys of the same JSON line (measured before the headline so that the GPU is warm when it starts):
  variants   other kernel instantiations at B=4,096 and B=65,536 (SPARSE_TRUE, f+grad+g, g, g+J)
  c3         one fixed sweep of 65,536 landing problems (per-problem x0), sharded over the ranks: STRONG scaling
  c4         ragged batch of 32,768 problems of 12 (N, k_trans, init_mode) classes per GPU
  c5         2^20 / 8 = 131,072 trajectories per GPU (37.4 GB of outputs per launch)
Rank 0 prints ONE JSON line.  The oracle (oracle/) is used here only as the timed CPU baseline and as the checker of
sampled results outside every timed region.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np

_emit = print
METRIC = "batched NLP evals/s (g+sparse Jacobian)"
UNIT = "evals/s"
B_PER_GPU = 4096
N_INPUT_SETS = 4            # 4 x 39.8 MB of decision vectors = 159 MB > 126 MB L2
SEED = 4096
SIGMA = 1e-2
HBM_FALLBACK_GBS = 6650.0   # /opt/skills/guides/B200_PROFILING.md fallback
BYTES_FULL = 285480         # SURVEY.md 8d: Z 9,720 + g 8,744 + grad 9,720 + f 8 + J 257,288
KERNEL = "ql::eval_kernel<1, 1, 0>"     # JM_BLOCK, reciprocal-FMA division, strided rows (as ncu / cuobjdump print it)
C4_CLASSES = [(N, kt, im) for (N, kt) in [(31, 11), (41, 14), (61, 21), (81, 27), (101, 34), (121, 41)] for im in (1, 2)]
DUMP_ROWS = 128             # --dump-outputs: 128 x (1215 + 1093 + 32161) doubles = 35 MB per dump
DUMP_SEED = 0


def workload_config(n_gpus):
    """Identical for both arms (the driver compares the two `config` objects)."""
    return {
        "workload": "C2: B=4096 perturbed decision vectors per GPU of the reference landing NLP "
                    "(N=61, k_trans=21, init_mode=1), Z_b = base[b mod 7] + 1e-2*xi_b, seed 4096",
        "outputs": "f, grad_f, g, SPARSE_BLOCK Jacobian values (full evaluation)",
        "jacobian_pattern": "SPARSE_BLOCK (32161 values/eval, reference column-major order)",
        "batch_per_gpu": B_PER_GPU,
        "global_batch": B_PER_GPU * n_gpus,
        "bytes_per_eval": BYTES_FULL,
        "l2": f"inputs rotate over {N_INPUT_SETS} distinct batches (159 MB > 126 MB L2); every step also writes 1.17 GB",
        "parallelism": f"batch sharded over {n_gpus} GPU(s), no collective on the hot path",
    }


def make_inputs(prob, rank, nsets):
    """Synthetic C2 batches (SURVEY.md 8d): bases = initial guess + the six shipped solutions."""
    import quadruped_landing_b200 as ql
    g = np.load(os.path.join(ROOT, "tests", "golden", "ref_solutions.npz"))
    bases = [ql.initial_guess(prob)] + [g[f"data_{i}"] for i in range(1, 7)]
    out = []
    for s in range(nsets):
        rng = np.random.default_rng(SEED + 1000 * rank + s)
        Z = np.stack([bases[b % 7] for b in range(B_PER_GPU)]) + SIGMA * rng.standard_normal((B_PER_GPU, prob.n_nlp))
        Z[:, 19::20] = np.clip(Z[:, 19::20], 1e-3, 2e-2)
        out.append(np.ascontiguousarray(Z))
    return out


def dump_outputs(path, outs):
    """Writes what one step returned to the caller as float64 DIR/<name>.npy: f for every evaluation of the batch;
    grad, g and jac for a fixed seeded sample of DUMP_ROWS evaluations (the whole Jacobian is 1.05 GB), whose batch
    indices go to rows.npy.  Inputs are seeded too, so two builds can be compared file by file."""
    rows = np.sort(np.random.default_rng(DUMP_SEED).choice(len(outs["f"]), DUMP_ROWS, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "rows.npy"), rows.astype(np.float64))
    for k, v in outs.items():
        if not isinstance(v, np.ndarray):                   # a CUDA tensor: gather the sampled rows on the device
            import torch
            v = (v if k == "f" else v[torch.from_numpy(rows).to(v.device)]).cpu().numpy()
        elif k != "f":
            v = v[rows]
        np.save(os.path.join(path, f"{k}.npy"), np.ascontiguousarray(v, dtype=np.float64))


class ClockSampler:
    """Polls NVML for SM clock and throttle reasons while the timed region runs."""

    def __init__(self, index, uuid=None):
        self.samples, self.reasons, self._stop = [], set(), threading.Event()
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            try:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(uuid)).encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
        self.t = threading.Thread(target=self._run, daemon=True)

    def _once(self):
        nv = self.nv
        self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
        r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
            else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
                 0x80: "hw_power_brake_slowdown"}
        for bit, name in names.items():
            if r & bit:
                self.reasons.add(name)

    def _run(self):
        while not self._stop.is_set():
            try:
                self._once()
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nv:
            self.t.start()

    def stop(self):
        if not self.nv:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"]}
        try:
            self._once()          # at least one sample while work is still queued / just finished
        except Exception:
            pass
        self._stop.set()
        self.t.join(timeout=1)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


def recorded_traffic():
    """dram bytes per launch of the dominant kernel from the committed ncu capture (profiles/), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f)
    except Exception:
        return None


def host_cores():
    """Threads the CPU baseline uses: every core this process may run on (torchrun exports OMP_NUM_THREADS=1,
    so the OpenMP default is not trusted; the count is passed to the oracle's num_threads clause)."""
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


class CpuRunner:
    """The CPU restatement (oracle port) on the host cores: all four outputs, SPARSE_BLOCK Jacobian.
    Buffers are allocated and first-touched once; step() times one pass over the batch."""

    def __init__(self, prob, Z, nthreads):
        from oracle import oracle as om
        self.o = om.Oracle(prob)
        o, n = self.o, Z.shape[0]
        self.n = n
        self.bufs = (np.empty(n), np.empty((n, o.n_nlp)), np.empty((n, o.m_nlp)), np.empty((n, o.nnz)))
        f, grad, g, jac = self.bufs
        self.Z = Z
        self.L = om.lib()
        self.args = (o.plan, o._p, n, om._ptr(Z), o.n_nlp, None, None, om._ptr(f), om._ptr(grad), o.n_nlp,
                     om._ptr(g), o.m_nlp, om._ptr(jac), o.nnz, int(nthreads))
        self.L.qlo_eval_batch(*self.args)              # first touch of the output pages

    def step(self):
        t0 = time.perf_counter()
        self.L.qlo_eval_batch(*self.args)
        return time.perf_counter() - t0


CPU_NOTE = ("CPU restatement of the reference algorithm (dense 20-wide forward-mode duals per knot), not Julia: "
            "no julia binary exists in the image.  The only recorded Julia figure is ~23 evals/s, 1 thread "
            "(src/main.ipynb:717-725).")


def run_reference(args):
    """--impl reference: the reference's algorithm on the host cores.  Julia is not installed in the image
    (DESIGN.md), so this is the C restatement in oracle/ (kind "port") with OpenMP over the batch.  Every step
    evaluates ALL 4,096 decision vectors of the batch; the run is bounded by the number of steps, not by sampling."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import quadruped_landing_b200 as ql
    prob = ql.default_problem()
    Z = make_inputs(prob, 0, 1)[0]
    cores = host_cores()
    runner = CpuRunner(prob, Z, cores)
    nwarm = 0
    for _ in range(max(0, args.warmup)):
        runner.step()
        nwarm += 1
        if nwarm >= 3:                                   # a CPU loop has no clocks to ramp: 3 passes warm the caches
            break
    times = [runner.step() for _ in range(args.steps)]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(zip(("f", "grad", "g", "jac"), runner.bufs)))
    value = B_PER_GPU * len(times) / sum(times)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": len(times), "warmup": nwarm, "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"all {B_PER_GPU} decision vectors of the batch per step, {len(times)} steps, "
                                   "OpenMP static schedule over the batch, outputs written to host memory"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": CPU_NOTE,
    }
    _emit(json.dumps(line))


# ------------------------------------------------------------------------------------------------ GPU arm
class Ctx:
    """What every section of the GPU arm needs."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the framework has no CPU path (use --impl reference for the CPU baseline)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.peak, self.peak_src = measured_peak()
        self.args = args

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, x):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())

    def timed(self, fn, steps, warmup=3):
        """`steps` calls of fn(i) between two CUDA events on the current stream, barrier + synchronize on both sides,
        max over ranks; returns ms per step."""
        torch = self.torch
        for i in range(warmup):
            fn(i)
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1)) / steps

    def roofline(self, bytes_per_launch, ms, kernel, launches_per_step=1):
        achieved = bytes_per_launch / (ms * 1e-3) / 1e9
        return {"bound": "hbm", "achieved": achieved, "peak": self.peak, "unit": "GB/s", "frac": achieved / self.peak,
                "traffic": None, "kernel": kernel, "peak_source": self.peak_src,
                "algorithmic_bytes_per_launch": bytes_per_launch / launches_per_step}


def padded(torch, Z, dev):
    """rows padded to an even length: 16-byte aligned rows let the kernel fetch a vector with one TMA load"""
    zp = torch.zeros((Z.shape[0], Z.shape[1] + 1), dtype=torch.float64, device=dev)
    zp[:, :Z.shape[1]] = Z if isinstance(Z, torch.Tensor) else torch.from_numpy(Z).to(dev)
    return zp[:, :Z.shape[1]]


def sample_check(nlp, out, Zrows, idx, x0=None, pattern="block"):
    """rows `idx` of a device result against the oracle (outside every timed region); returns "ok" or a message"""
    from oracle.oracle import Oracle
    torch_idx = out["jac"].new_tensor(idx, dtype=__import__("torch").int64)
    ref = Oracle(nlp.prob).eval_batch(Zrows, x0=x0, want=tuple(k for k in ("f", "grad", "g", "jac") if k in out), pattern=pattern)
    for k, r in ref.items():
        got = out[k][torch_idx].cpu().numpy()
        if not np.all(np.abs(got - r) <= 1e-14 + 1e-12 * np.abs(r)):
            return f"{k}: outside 1e-12 relative / 1e-14 absolute"
    return "ok"


def section_variants(cx, prob, host_sets):
    """Other kernel instantiations (SPARSE_TRUE pattern, no Jacobian, g + J), device-resident, B=4,096 and 65,536."""
    import quadruped_landing_b200 as ql
    torch = cx.torch
    res = []
    nb, nt = ql.HybridNLP.from_problem(prob, device=cx.local), ql.HybridNLP.from_problem(prob, pattern="true", device=cx.local)
    n, m = nb.n_nlp, nb.m_nlp
    cases = [("SPARSE_TRUE f+grad+g+J", nt, ("f", "grad", "g", "jac"), 8 * (2 * n + m + 1 + nt.nnz), "ql::eval_kernel<2, 1, 0>"),
             ("f+grad+g (no Jacobian)", nb, ("f", "grad", "g"), 8 * (2 * n + m + 1), "ql::eval_kernel<0, 1, 0>"),
             ("g only", nb, ("g",), 8 * (n + m), "ql::eval_kernel<0, 1, 0>"),
             ("SPARSE_BLOCK g+J", nb, ("g", "jac"), 8 * (n + m + nb.nnz_block), "ql::eval_kernel<1, 1, 0>"),
             ("SPARSE_BLOCK f+grad+g+J", nb, ("f", "grad", "g", "jac"), BYTES_FULL, "ql::eval_kernel<1, 1, 0>")]
    for B in (B_PER_GPU, 65536):
        reps = -(-B // B_PER_GPU)
        # distinct inputs larger than L2 at both sizes: 4 sets of 4,096 or one batch of 65,536 (637 MB)
        if B == B_PER_GPU:
            Zs = [padded(torch, z, cx.dev) for z in host_sets]
        else:
            Zs = [padded(torch, torch.from_numpy(np.concatenate(host_sets)).to(cx.dev).repeat(reps // len(host_sets), 1), cx.dev)]
        for name, nlp, want, nbytes, kern in cases:
            if B == B_PER_GPU and name == "SPARSE_BLOCK f+grad+g+J":
                continue                                    # that is the headline
            out = nlp.eval_batch(Zs[0], want=want)
            steps = 40 if B == B_PER_GPU else 10
            ms = cx.timed(lambda i: nlp.eval_batch(Zs[i % len(Zs)], want=want, out=out), steps)
            r = cx.roofline(nbytes * B, ms, kern)
            res.append({"what": name, "batch_per_gpu": B, "value": B * cx.world / (ms * 1e-3), "unit": UNIT,
                        "ms_per_launch": ms, "bytes_per_eval": nbytes, "GBps_per_gpu": r["achieved"], "frac": r["frac"],
                        "kernel": kern, "warps_per_sm": nlp.launch_info()["blocks_per_sm"]})
            del out
        del Zs
        torch.cuda.empty_cache()
    return res


def section_c3(cx, prob):
    """SURVEY.md 8d C3: ONE fixed sweep of 65,536 landing problems (256 drop heights x 256 initial pitches, per-problem
    x0), all four outputs per iteration, 10 iterations with Z += 1e-3 xi, sharded contiguously over the ranks
    (strong scaling).  Sharding goes through sharding.evaluate_sharded (NCCL all-gather of f after the timed region)."""
    import quadruped_landing_b200 as ql
    torch, dist = cx.torch, cx.dist
    B = 65536
    nlp = ql.HybridNLP.from_problem(prob, device=cx.local)
    x0_all = ql.sweep_initial_states(prob.model, np.linspace(0.25, 3.0, 256), np.linspace(-40.0, -5.0, 256))
    lo, hi = ql.shard_bounds(B, cx.world, cx.rank)
    x0d = torch.from_numpy(x0_all[lo:hi]).to(cx.dev)
    Z = nlp.initial_guess_batch(x0d)                        # guesses built on the device (rows padded to an even length)
    gen = torch.Generator(device=cx.dev).manual_seed(3 + cx.rank)
    noise = 1e-3 * torch.randn((hi - lo, nlp.n_nlp), generator=gen, device=cx.dev, dtype=torch.float64)
    out = nlp.eval_batch(Z, x0=x0d)
    iters = 10
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]

    def it(i):
        kev[i][0].record()
        nlp.eval_batch(Z, x0=x0d, out=out)
        kev[i][1].record()
        Z.add_(noise)                                       # the "iteration": perturb every decision vector

    ms = cx.timed(it, iters, warmup=2)                      # ms per iteration (evaluation + perturbation), max over ranks
    ms_kernel = cx.max_over_ranks(sum(a.elapsed_time(b) for a, b in kev) / iters)      # the evaluator's launch alone
    # correctness + the sharded entry point, outside the timed region: every rank evaluates its slice of the GLOBAL
    # batch through evaluate_sharded and the objectives are all-gathered over NCCL
    x0g = torch.from_numpy(x0_all).to(cx.dev)
    Zg = nlp.initial_guess_batch(x0g)
    lo_hi = {}

    def evaluate(Zl):
        l, h = ql.shard_bounds(B, cx.world, cx.rank)
        lo_hi["b"] = (l, h)
        return nlp.eval_batch(padded(torch, Zl, cx.dev), x0=x0g[l:h], want=("f", "g"))

    _, (l2, h2), fall = ql.evaluate_sharded(evaluate, Zg, gather="f")
    torch.cuda.synchronize()
    check = "ok"
    if cx.rank == 0:
        from oracle.oracle import Oracle
        idx = np.arange(0, B, 1021)
        ref = Oracle(prob).eval_batch(Zg[torch.from_numpy(idx).to(cx.dev)].cpu().numpy(), x0=x0_all[idx], want=("f",))
        if fall.shape[0] != B or not np.array_equal(fall[torch.from_numpy(idx).to(cx.dev)].cpu().numpy(), ref["f"]):
            check = "gathered objectives differ from the oracle"
    nbytes = (BYTES_FULL + 240) * (hi - lo)                 # + per-problem x0/xf stream (SURVEY 8d)
    r = cx.roofline(nbytes, ms_kernel, KERNEL)
    res = {"workload": "C3: fixed sweep of 65,536 landing problems (256 drop heights x 256 pitches, per-problem x0), "
                       "10 iterations of f+grad+g+J with Z += 1e-3 xi in between, contiguous shards",
           "scaling": "strong", "global_batch": B, "batch_per_gpu": hi - lo, "iterations": iters,
           "value": B / (ms * 1e-3), "unit": UNIT, "ms_per_iteration": ms, "ms_per_evaluator_launch": ms_kernel,
           "roofline": r, "gpu_launches": iters * cx.world,
           "sharded_check": check, "sharded_via": "sharding.evaluate_sharded + NCCL all_gather of f (outside the timed region)"}
    del out, Z, Zg, noise
    torch.cuda.empty_cache()
    return res


def section_c4(cx):
    """SURVEY.md 8d C4: ragged batch, 12 (N, k_trans, init_mode) classes uniformly mixed, B=32,768 per GPU, seed 7."""
    import quadruped_landing_b200 as ql
    torch = cx.torch
    probs = [ql.build_problem(N=N, k_trans=kt, init_mode=im) for N, kt, im in C4_CLASSES]
    ev = ql.RaggedEvaluator(probs, device=cx.local)
    rng = np.random.default_rng(7 + cx.rank)
    B = 32768
    class_of = rng.integers(0, len(probs), size=B)
    off = ev.offsets(class_of)
    guesses = [ql.initial_guess(p) for p in probs]
    vecs = []
    for c in class_of:
        v = guesses[c] + 1e-2 * rng.standard_normal(probs[c].n_nlp)
        v[19::20] = np.clip(v[19::20], 1e-3, 2e-2)
        vecs.append(v)
    Zd = torch.from_numpy(ev.pack(class_of, vecs)).to(cx.dev)
    plan = ev.plan(class_of, cx.dev)
    out = ev.eval(plan, Zd)
    ms = cx.timed(lambda i: ev.eval(plan, Zd, out=out), 5, warmup=2)
    nbytes = 8 * int(sum(2 * ev.n[c] + ev.m[c] + ev.nnz[c] + 1 for c in class_of))
    r = cx.roofline(nbytes, ms, "ql::eval_kernel<1, 1, 1>", launches_per_step=len(probs))
    check = "ok"
    if cx.rank == 0:
        from oracle.oracle import Oracle
        for b in range(0, B, 2731):
            c = class_of[b]
            e = ev.nlps[c]
            ref = Oracle(probs[c]).eval_batch(vecs[b][None, :])
            got = {"f": out["f"][b:b + 1], "grad": out["grad"][off["z_off"][b]:off["z_off"][b] + e.n_nlp],
                   "g": out["g"][off["g_off"][b]:off["g_off"][b] + e.m_nlp],
                   "jac": out["jac"][off["j_off"][b]:off["j_off"][b] + e.nnz_block]}
            for k, v in got.items():
                a, w = v.cpu().numpy().reshape(-1), ref[k].reshape(-1)
                if not np.all(np.abs(a - w) <= 1e-14 + 1e-12 * np.abs(w)):
                    check = f"problem {b} {k}: outside tolerance"
    res = {"workload": "C4: ragged batch of 32,768 problems per GPU, 12 classes (N, k_trans) in {(31,11),(41,14),(61,21),"
                       "(81,27),(101,34),(121,41)} x init_mode in {1,2} uniformly mixed, flat arrays + offset tables",
           "scaling": "weak", "batch_per_gpu": B, "value": B * cx.world / (ms * 1e-3), "unit": UNIT, "ms_per_pass": ms,
           "bytes_per_pass": nbytes, "roofline": r, "gpu_launches": 5 * ev.launches_per_eval * cx.world, "oracle_check": check,
           "launches_per_pass": ev.launches_per_eval}
    del out, Zd
    torch.cuda.empty_cache()
    return res


def section_c5(cx, prob):
    """SURVEY.md 8d C5: 2^20 perturbed copies of Z0 over 8 GPUs = 131,072 per GPU, sigma = 5e-2, full evaluation
    (37.4 GB of outputs per launch per GPU)."""
    import quadruped_landing_b200 as ql
    torch = cx.torch
    B = 131072
    nlp = ql.HybridNLP.from_problem(prob, device=cx.local)
    gen = torch.Generator(device=cx.dev).manual_seed(2 ** 20 + cx.rank)
    Z = torch.zeros((B, nlp.n_nlp + 1), dtype=torch.float64, device=cx.dev)[:, :nlp.n_nlp]
    Z.copy_(torch.from_numpy(ql.initial_guess(prob)).to(cx.dev)[None, :] +
            5e-2 * torch.randn((B, nlp.n_nlp), generator=gen, device=cx.dev, dtype=torch.float64))
    Z[:, 19::20].clamp_(1e-3, 2e-2)
    out = nlp.eval_batch(Z)
    steps = 3
    ms = cx.timed(lambda i: nlp.eval_batch(Z, out=out), steps, warmup=1)
    check = "ok"
    if cx.rank == 0:
        idx = np.arange(0, B, 4099)
        check = sample_check(nlp, out, Z[torch.from_numpy(idx).to(cx.dev)].cpu().numpy(), idx)
    r = cx.roofline(BYTES_FULL * B, ms, KERNEL)
    res = {"workload": "C5: 2^20-trajectory multi-start batch over 8 GPUs = 131,072 perturbed copies of Z0 per GPU "
                       "(sigma 5e-2), f+grad+g+J, 37.4 GB of outputs per launch per GPU",
           "scaling": "weak", "batch_per_gpu": B, "global_batch": B * cx.world, "value": B * cx.world / (ms * 1e-3),
           "unit": UNIT, "ms_per_launch": ms, "roofline": r, "gpu_launches": steps * cx.world, "oracle_check": check}
    del out, Z
    torch.cuda.empty_cache()
    return res


def pcie_and_host_ceilings(cx, nlp, jac_host):
    """The two ceilings of the host-pointer path, measured here: D2H copy bandwidth from the GPU into pinned memory,
    and what the handle's worker pool writes into the caller's rows with non-temporal stores (timed on
    qlnlp_host_output_register, which writes the constant image of every row)."""
    torch = cx.torch
    n = 1 << 28
    d = torch.empty(n, dtype=torch.uint8, device=cx.dev)
    h = torch.empty(n, dtype=torch.uint8).pin_memory()
    h.copy_(d, non_blocking=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(4):
        h.copy_(d, non_blocking=True)
    torch.cuda.synchronize()
    d2h = 4 * n / (time.perf_counter() - t0) / 1e9
    del d, h
    nlp.register_host_output(jac_host)
    cx.barrier()                                   # every rank streams at the same time: they share the host's memory
    t0 = time.perf_counter()
    nlp.register_host_output(jac_host)
    host_w = jac_host.nbytes / (time.perf_counter() - t0) / 1e9
    cx.barrier()
    return d2h, host_w


def run_gpu(args):
    import quadruped_landing_b200 as ql
    cx = Ctx(args)
    torch, dist = cx.torch, cx.dist
    world, rank, local, dev = cx.world, cx.rank, cx.local, cx.dev
    n_gpus = world

    prob = ql.default_problem()
    nlp = ql.HybridNLP.from_problem(prob, device=local)
    host_sets = make_inputs(prob, rank, N_INPUT_SETS)
    extras = {}

    def guarded(name, fn):
        """An extra must never cost the headline: its failure is recorded, not raised (all ranks fail alike)."""
        try:
            extras[name] = fn()
        except Exception as e:                               # noqa: BLE001
            extras[name] = {"error": f"{type(e).__name__}: {e}"[:300]}
            torch.cuda.synchronize()
            torch.cuda.empty_cache()

    # ---- extras first: they also bring the GPU to its working clocks before the headline starts
    if not args.no_extras:
        skip = set(os.environ.get("QL_BENCH_SKIP", "").split(","))      # diagnosis only: leave sections out
        for name, fn in (("variants", lambda: section_variants(cx, prob, host_sets)), ("c3", lambda: section_c3(cx, prob)),
                         ("c4", lambda: section_c4(cx)), ("c5", lambda: section_c5(cx, prob))):
            if name not in skip:
                guarded(name, fn)

    # ---- headline: device-resident throughput of C2 ---------------------------------------------------------
    Zs = [padded(torch, z, dev) for z in host_sets]
    want = ("f", "grad", "g", "jac")
    out = nlp.eval_batch(Zs[0], want=want)
    torch.cuda.synchronize()
    for i in range(args.warmup):                             # exactly W warm-up steps, as asked
        nlp.eval_batch(Zs[i % N_INPUT_SETS], want=want, out=out)
    sampler = ClockSampler(local, getattr(torch.cuda.get_device_properties(local), "uuid", None))
    cx.barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(args.steps):
        nlp.eval_batch(Zs[s % N_INPUT_SETS], want=want, out=out)
    e1.record()
    cx.barrier()
    clocks = sampler.stop()
    ms_step = cx.max_over_ranks(e0.elapsed_time(e1)) / args.steps
    value = B_PER_GPU * n_gpus / (ms_step * 1e-3)
    launch_info = nlp.launch_info()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)                 # rank 0's batch of the last timed step

    # ---- end to end through the C ABI with HOST buffers (pinned), copies inside the timed region -----------------
    # caller-side arrays come from the library's allocator (qlnlp_host_alloc: page-locked, 2 MB pages where granted)
    def pinned(shape):
        try:
            return ql.host_alloc(shape)
        except Exception:                                    # noqa: BLE001
            return torch.empty(shape, dtype=torch.float64).pin_memory().numpy()

    class _Pin:                                              # the two input batches the host calls alternate between
        def __init__(self, z):
            self.a = pinned(z.shape)
            self.a[:] = z

        def numpy(self):
            return self.a

    pin = [_Pin(z) for z in host_sets[:2]]
    hnp = {"f": pinned((B_PER_GPU,)), "grad": pinned((B_PER_GPU, nlp.n_nlp)), "g": pinned((B_PER_GPU, nlp.m_nlp)),
           "jac": pinned((B_PER_GPU, nlp.nnz_block))}
    e2e_steps = max(3, min(args.steps, 20))

    def time_host(ev, outs, wanted=want, label=""):
        for s in range(3):
            ev.eval_batch_host(pin[s % 2].numpy(), want=wanted, out=outs)
        best = None
        for attempt in range(2):       # the host's memory system is shared with other tenants: best of two passes
            cx.barrier()
            tt0 = ev._debug_host_times()
            t0 = time.perf_counter()
            for s in range(e2e_steps):
                ev.eval_batch_host(pin[s % 2].numpy(), want=wanted, out=outs)
            torch.cuda.synchronize()
            t = cx.max_over_ranks(time.perf_counter() - t0)
            tt1 = ev._debug_host_times()
            cx.barrier()
            if rank == 0:
                print(f"[bench] host path {label} pass {attempt}: {t / e2e_steps * 1e3:.2f} ms per call; library: " +
                      ", ".join(f"{k} {(tt1[k] - tt0[k]) / e2e_steps * 1e3:.2f}" for k in tt0), file=sys.stderr)
            best = t if best is None else min(best, t)
        return B_PER_GPU * n_gpus * e2e_steps / best

    e2e_unreg = time_host(nlp, hnp, label="unregistered")     # every 64-byte line of every row rewritten
    d2h_gbs, host_w_gbs = pcie_and_host_ceilings(cx, nlp, hnp["jac"])      # also registers the output rows
    e2e_value = time_host(nlp, hnp, label="registered")       # registered rows: only the lines that change
    # exactness of what the timed calls produced: host rows == device rows, bit for bit (outside the timed region)
    dref = nlp.eval_batch(padded(torch, pin[(e2e_steps - 1) % 2].numpy(), dev), want=want)
    torch.cuda.synchronize()
    e2e_check = "ok" if all(np.array_equal(hnp[k], dref[k].cpu().numpy()) for k in want) else "host rows differ from device rows"
    del dref
    info = nlp.host_path_info()
    h2d = B_PER_GPU * nlp.n_nlp * 8
    d2h = B_PER_GPU * (1 + nlp.n_nlp + nlp.m_nlp + nlp.nnz_block) * 8
    pcie_d2h = B_PER_GPU * (1 + nlp.n_nlp + nlp.m_nlp + info["pcie_jac_doubles_per_eval"]) * 8
    host_bytes = B_PER_GPU * info["touched_lines_per_row"] * 64
    # Ceiling of the registered path: the slower of PCIe (D2H of 41 KB per evaluation) and HOST MEMORY, which sees
    # every byte of the step once more than PCIe does: the DMA writes (D2H) and reads (H2D), the row builder reading
    # the staged values and writing the touched lines.
    stage_bytes = B_PER_GPU * info["pcie_jac_doubles_per_eval"] * 8
    host_traffic = pcie_d2h + h2d + stage_bytes + host_bytes
    # per-rank bandwidths were measured with all ranks active; the node's ceiling is the sum over the ranks
    host_w_node = cx.sum_over_ranks(host_w_gbs)
    t_pcie, t_host = pcie_d2h / (d2h_gbs * 1e9), host_traffic / (host_w_gbs * 1e9)
    e2e_ceiling = B_PER_GPU / max(t_pcie, t_host)
    e2e_ceiling_node = cx.sum_over_ranks(e2e_ceiling)
    nlp.unregister_host_output(hnp["jac"])
    nlp_t = ql.HybridNLP.from_problem(prob, pattern="true", device=local)
    hnp_t = dict(hnp, jac=pinned((B_PER_GPU, nlp_t.nnz)))
    e2e_true = time_host(nlp_t, hnp_t, label="SPARSE_TRUE rows")
    del nlp_t, hnp_t

    # ---- optional final gather of per-problem scalars over NCCL (outside every timed region)
    if world > 1:
        parts = [torch.empty_like(out["f"]) for _ in range(world)]
        dist.all_gather(parts, out["f"])
        torch.cuda.synchronize()

    # ---- single process driving several GPUs through the C ABI (qlnlp_create_multi): rank 0 only, others wait
    multi = None
    if world > 1 and not args.no_extras:
        cx.barrier()
        if rank == 0:
            try:
                mh = ql.HybridNLP.from_problem(prob, devices=list(range(world)))
                mh.set_option("host_threads", max(1, host_cores() // world))     # the other ranks are idle: all cores
                Bm = B_PER_GPU * world
                Zm = pinned((Bm, nlp.n_nlp))
                Zm[:] = np.concatenate([host_sets[i % N_INPUT_SETS] for i in range(world)])
                om = {"f": pinned((Bm,)), "grad": pinned((Bm, nlp.n_nlp)), "g": pinned((Bm, nlp.m_nlp)),
                      "jac": pinned((Bm, nlp.nnz_block))}
                mh.register_host_output(om["jac"])
                for _ in range(2):
                    mh.eval_batch_host(Zm, out=om)
                t0 = time.perf_counter()
                for _ in range(5):
                    mh.eval_batch_host(Zm, out=om)
                tm = (time.perf_counter() - t0) / 5
                dchk = nlp.eval_batch(padded(torch, Zm[Bm - 64:], dev), want=("jac", "g"))      # the last shard's rows, on this rank's GPU
                torch.cuda.synchronize()
                ok = np.array_equal(om["jac"][Bm - 64:], dchk["jac"].cpu().numpy()) and np.array_equal(om["g"][Bm - 64:], dchk["g"].cpu().numpy())
                multi = {"what": "ONE host thread, ONE qlnlp_eval_batch_host call on a multi-device handle "
                                 "(qlnlp_create_multi): the library shards the batch over the GPUs (registered rows)",
                         "devices": world, "global_batch": Bm, "value": Bm / tm, "unit": UNIT, "ms_per_call": tm * 1e3,
                         "check": "ok" if ok else "rows differ from a single-device evaluation",
                         "threads_per_device": mh.host_path_info()["threads_per_device"]}
                del mh, om, Zm
            except Exception as e:                           # noqa: BLE001
                multi = {"error": f"{type(e).__name__}: {e}"[:300]}
        cx.barrier()

    if rank == 0:
        bytes_per_launch = BYTES_FULL * B_PER_GPU
        achieved = bytes_per_launch / (ms_step * 1e-3) / 1e9          # GB/s per GPU (max-over-ranks time)
        traffic = recorded_traffic()
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(n_gpus),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "passes": "best of 2 passes of `steps` calls", "check": e2e_check,
                    "path": "qlnlp_eval_batch_host on page-locked host buffers (qlnlp_host_alloc), output rows registered once "
                            "(qlnlp_host_output_register, like jac_c! relying on the caller's zeros): 512-evaluation chunks "
                            "pipelined over 4 streams; f/grad/g land in the caller's arrays by DMA; of the 32,161 SPARSE_BLOCK "
                            "values per evaluation only the 2,794 value-dependent ones cross PCIe and a persistent pool of host "
                            "threads rewrites the 64-byte lines that hold them (non-temporal AVX-512 stores, no arithmetic)",
                    "pcie_d2h_bytes_per_step": pcie_d2h, "host_bytes_written_per_step": host_bytes,
                    "host_threads": info["threads_per_device"], "avx512": bool(info["avx512"]),
                    "roofline": {"bound": "pcie_d2h" if t_pcie >= t_host else "host_dram",
                                 "pcie_d2h_GBps_measured": d2h_gbs, "host_dram_GBps_measured": host_w_gbs,
                                 "host_memory_bytes_per_step": host_traffic,
                                 "host_dram_GBps_node": host_w_node,
                                 "ceiling_evals_per_s_per_gpu": e2e_ceiling, "ceiling_evals_per_s_node": e2e_ceiling_node,
                                 "frac": e2e_value / e2e_ceiling_node,
                                 "how": "ceiling = 4096 / max(PCIe D2H bytes / measured D2H copy bandwidth, host-memory bytes / "
                                        "host bandwidth); host-memory bytes = DMA writes + DMA reads + staged values read by the row "
                                        "builder + 64-byte lines it rewrites; host bandwidth = what this handle's worker pool reaches "
                                        "streaming whole rows with non-temporal stores (qlnlp_host_output_register timed on the "
                                        "1 GB output array); both measured in this run, with every rank streaming at the same time "
                                        "(the ranks of a node share its memory system), summed over the ranks for the node ceiling"},
                    "unregistered": {"value": e2e_unreg, "unit": UNIT,
                                     "what": "same call without registration: every line of every row rewritten (257 KB per evaluation)"},
                    "sparse_true": {"value": e2e_true, "unit": UNIT,
                                    "what": "SPARSE_TRUE handle (4,840 values per evaluation), unregistered rows"}},
            "gpu_launches": args.steps * n_gpus,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": cx.peak, "unit": "GB/s", "frac": achieved / cx.peak,
                         "traffic": (traffic or {}).get("dram_bytes_per_launch"),
                         "kernel": KERNEL, "peak_source": cx.peak_src,
                         "algorithmic_bytes_per_launch": bytes_per_launch,
                         "traffic_source": (traffic or {}).get("source")},
            "launch": launch_info,
        }
        line.update(extras)
        if multi is not None:
            line["c_abi_multi_gpu"] = multi
        # CPU baseline beside it (rank 0): bounded sample of the same batch
        if not args.no_cpu:
            cores = host_cores()
            sample = B_PER_GPU if n_gpus == 1 else 1024
            runner = CpuRunner(prob, host_sets[0][:sample], cores)
            v = sample / statistics.median([runner.step() for _ in range(3)])
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": f"{sample} decision vectors of the same batch, 3 repetitions (median), "
                                              "OpenMP over the batch on all host cores" +
                                              ("" if n_gpus == 1 else f" (shared with {n_gpus - 1} waiting ranks)"),
                                    "note": CPU_NOTE}
        _emit(json.dumps(line))
    if world > 1:
        cx.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extras", action="store_true", help="headline + e2e only (what the ncu captures run)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    # the contract is ONE JSON line on stdout: libraries (e.g. NCCL's version banner) also write to fd 1, so
    # point fd 1 at stderr while running and emit the line on the real stdout at the end
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    global _emit
    _emit = lambda line: os.write(real_stdout, (line + "\n").encode())
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
