"""Ragged batches: problems of mixed horizon / contact schedule in one call (SURVEY.md 8d, config C4).

The reference has a single problem size per `HybridNLP`; "varying horizon" sweeps therefore mix several
(N, k_trans, init_mode) classes.  Each class gets its own handle (its own segment plan and cost tables); the
whole mixed batch is evaluated by ONE fused launch (`qlnlp_eval_ragged_classes`): problems are handed out
ordered by class, largest horizon first, and a warp swaps class records when the class changes.  Inputs and
outputs are flat arrays with offset tables, the layout C4 asks for.
"""
from __future__ import annotations

from typing import Dict, List, Sequence

import numpy as np

from .evaluator import HybridNLP, _device_empty
from .problem import ProblemData


class RaggedEvaluator:
    """Evaluates a batch whose b-th problem belongs to class ``class_of[b]`` (index into ``probs``)."""

    def __init__(self, probs: Sequence[ProblemData], device: int = 0):
        self.probs = list(probs)
        self.nlps: List[HybridNLP] = [HybridNLP.from_problem(p, device=device) for p in self.probs]
        self.device = device
        self.n = np.array([e.n_nlp for e in self.nlps], dtype=np.int64)
        self.m = np.array([e.m_nlp for e in self.nlps], dtype=np.int64)
        self.nnz = np.array([e.nnz_block for e in self.nlps], dtype=np.int64)
        self._plan = None
        self.launches_per_eval = 1                     # one fused launch for the whole mixed batch

    def offsets(self, class_of: np.ndarray) -> Dict[str, np.ndarray]:
        """Row starts (in doubles): problem b owns Z[z_off[b] : z_off[b] + n_b], g[g_off[b] : ...], jac[j_off[b] : ...].
        Every row is padded to an even length, so all rows are 16-byte aligned (TMA load / store paths); the last
        entry of each table is the total length to allocate."""
        class_of = np.asarray(class_of, dtype=np.int64)
        even = lambda w: (w + 1) & ~1
        cs = lambda w: np.concatenate([[0], np.cumsum(even(w)[class_of])])
        return {"z_off": cs(self.n), "g_off": cs(self.m), "j_off": cs(self.nnz)}

    def pack(self, class_of: np.ndarray, vectors) -> np.ndarray:
        """Lay decision vectors (one per problem) out in the padded flat Z layout of ``offsets``."""
        off = self.offsets(class_of)["z_off"]
        Z = np.zeros(int(off[-1]))
        for b, v in enumerate(vectors):
            Z[off[b]:off[b] + len(v)] = v
        return Z

    def plan(self, class_of: np.ndarray, device=None) -> "RaggedPlan":
        """Everything about a batch that does not depend on the decision vectors: the offset tables and the launch
        order, uploaded once.  ``eval`` caches the plan of the last ``class_of`` it saw, so repeated evaluations of
        one batch (solver iterations) do no per-call host work."""
        import torch

        class_of = np.ascontiguousarray(class_of, dtype=np.int64)
        dev = torch.device("cuda", self.device) if device is None else device
        off = self.offsets(class_of)
        doff = {k: torch.from_numpy(v).to(dev) for k, v in off.items()}
        # all problems, ordered by class, largest horizon first (the long evaluations start first)
        by_class = sorted(range(len(self.nlps)), key=lambda c: -self.nlps[c].N)
        rank_of = np.empty(len(self.nlps), dtype=np.int64)
        rank_of[by_class] = np.arange(len(self.nlps))
        order = np.argsort(rank_of[class_of], kind="stable")
        plan = RaggedPlan(class_of.copy(), off, doff)
        plan.order = torch.from_numpy(order.astype(np.int64)).to(dev)
        plan.dclass = torch.from_numpy(class_of.astype(np.int32)).to(dev)
        return plan

    def eval(self, class_of, Z_flat, want=("f", "grad", "g", "jac"), out=None):
        """``Z_flat``: 1-D float64 CUDA tensor holding the decision vectors back to back (see ``offsets``);
        ``class_of``: the class index of every problem, or a ``RaggedPlan``.  Returns flat CUDA tensors ``f[B]``,
        ``grad`` (Z layout), ``g``, ``jac`` and the offset tables; pass the returned dict back as ``out`` to reuse
        the output arrays.

        The whole mixed batch is ONE ``qlnlp_eval_ragged_classes`` launch; the kernel addresses each problem's rows
        through the offset tables, so nothing is gathered or scattered."""
        import torch

        dev = Z_flat.device
        if isinstance(class_of, RaggedPlan):
            plan = class_of
        else:
            class_of = np.ascontiguousarray(class_of, dtype=np.int64)
            plan = self._plan
            if plan is None or plan.class_of.shape != class_of.shape or not np.array_equal(plan.class_of, class_of):
                plan = self._plan = self.plan(class_of, dev)
        B = plan.class_of.shape[0]
        off = plan.off
        flat = {"Z": Z_flat}
        sizes = {"f": B, "grad": int(off["z_off"][-1]), "g": int(off["g_off"][-1]), "jac": int(off["j_off"][-1])}
        missing = []
        for name in ("f", "grad", "g", "jac"):
            if name in want:
                t = None if out is None else out.get(name)
                if t is None or t.numel() != sizes[name] or t.device != dev:
                    missing.append(name)
                else:
                    flat[name] = t
        if missing:                        # the library's output pool, compressible where the device offers it
            ts = _device_empty(dev.index, [(sizes[k], None, torch.float64) for k in missing], self.nlps[0]._compressible)
            flat.update(zip(missing, ts))
        HybridNLP.eval_ragged_classes(self.nlps, plan.order, plan.dclass, flat, plan.doff, z_padded=True)
        res = {k: v for k, v in flat.items() if k != "Z"}
        res.update(off)
        self._keep = plan                  # alive until the next call: the launches are asynchronous
        return res


class RaggedPlan:
    """Offset tables (host + device) and launch order of one mixed batch (``RaggedEvaluator.plan``)."""

    def __init__(self, class_of, off, doff):
        self.class_of, self.off, self.doff = class_of, off, doff
