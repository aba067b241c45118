#!/usr/bin/env python3
"""Generates quadruped_landing_b200/csrc/rk4_dual_gen.h.

What it does
------------
It symbolically executes the reference's RK4 step (src/planar_quadruped.jl:189-221
over the three vector fields :36-185) on forward-mode dual numbers seeded like
``ForwardDiff.jacobian(f, [x;u])`` (:225-248, one 20-wide chunk), with the dual
arithmetic rules of ForwardDiff 0.10.25 (the same rules oracle/ql_oracle.c applies
densely), but tracks which partials are STRUCTURALLY zero and drops every operation
whose result is exactly determined without rounding:

    x*0 -> 0      x*1 -> x      x+0 -> x      x-0 -> x      0-x -> -x
    0/c -> 0      const (op) const -> folded in IEEE double by Python

Every remaining operation is emitted in the reference's order with the reference's
operand pairing, as explicit round-to-nearest add/mul/div (no FMA contraction).  The
emitted straight-line code is therefore BIT-IDENTICAL to the dense dual evaluation
for finite inputs (up to the sign of zero), while doing ~1/10 of the arithmetic and
holding only the structurally non-zero Jacobian entries in registers.
(tests/test_rk4_gen.py checks the bit-identity against the oracle on the CPU.)

It also emits, per mode, the sparsity pattern of the 15x20 block and the code that
patches those entries into a knot's run of the SPARSE_BLOCK value stream.

Usage:  python tools/gen_rk4_dual.py            (rewrites the header in place)
"""
from __future__ import annotations

import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "..", "quadruped_landing_b200", "csrc", "rk4_dual_gen.h")

NX, NU, NP = 15, 5, 20


class Graph:
    """Hash-consed expression DAG over fp64 with exact-only simplifications."""

    def __init__(self):
        self.nodes = []          # id -> tuple
        self.index = {}          # tuple -> id
        self.zero = self.const(0.0)
        self.one = self.const(1.0)

    def _mk(self, key):
        i = self.index.get(key)
        if i is None:
            i = len(self.nodes)
            self.nodes.append(key)
            self.index[key] = i
        return i

    def const(self, v):
        v = float(v)
        if v == 0.0:
            v = 0.0  # collapse -0.0: the sign of zero is not part of parity
        return self._mk(("c", v))

    def inp(self, name):
        return self._mk(("in", name))

    def is_const(self, a):
        return self.nodes[a][0] == "c"

    def cval(self, a):
        return self.nodes[a][1]

    def add(self, a, b):
        if self.is_const(a) and self.is_const(b):
            return self.const(self.cval(a) + self.cval(b))
        if a == self.zero:
            return b
        if b == self.zero:
            return a
        if a > b:
            a, b = b, a  # IEEE add is commutative
        return self._mk(("add", a, b))

    def sub(self, a, b):
        if self.is_const(a) and self.is_const(b):
            return self.const(self.cval(a) - self.cval(b))
        if b == self.zero:
            return a
        if a == self.zero:
            return self.neg(b)
        return self._mk(("sub", a, b))

    def neg(self, a):
        if self.is_const(a):
            return self.const(-self.cval(a))
        if self.nodes[a][0] == "neg":
            return self.nodes[a][1]
        return self._mk(("neg", a))

    def mul(self, a, b):
        if self.is_const(a) and self.is_const(b):
            return self.const(self.cval(a) * self.cval(b))
        if a == self.zero or b == self.zero:
            return self.zero
        if a == self.one:
            return b
        if b == self.one:
            return a
        if self.is_const(a) and self.cval(a) == -1.0:
            return self.neg(b)
        if self.is_const(b) and self.cval(b) == -1.0:
            return self.neg(a)
        if a > b:
            a, b = b, a  # IEEE mul is commutative
        return self._mk(("mul", a, b))

    def div(self, a, b):
        if self.is_const(a) and self.is_const(b):
            return self.const(self.cval(a) / self.cval(b))
        if a == self.zero:
            return self.zero
        if b == self.one:
            return a
        return self._mk(("div", a, b))


class Dual:
    __slots__ = ("g", "v", "p")

    def __init__(self, g, v, p=None):
        self.g = g
        self.v = v
        self.p = {} if p is None else {j: n for j, n in p.items() if n != g.zero}

    def part(self, j):
        return self.p.get(j, self.g.zero)

    def _keys(self, o):
        return sorted(set(self.p) | set(o.p))

    # ForwardDiff dual.jl / partials.jl rules -------------------------------------------
    def add(self, o):
        g = self.g
        return Dual(g, g.add(self.v, o.v), {j: g.add(self.part(j), o.part(j)) for j in self._keys(o)})

    def sub(self, o):
        g = self.g
        return Dual(g, g.sub(self.v, o.v), {j: g.sub(self.part(j), o.part(j)) for j in self._keys(o)})

    def mul(self, y):
        # Dual(vx*vy, _mul_partials(px, py, vy, vx)):  (vy * px_i) + (vx * py_i)
        g, x = self.g, self
        return Dual(g, g.mul(x.v, y.v),
                    {j: g.add(g.mul(y.v, x.part(j)), g.mul(x.v, y.part(j))) for j in x._keys(y)})

    def neg(self):
        g = self.g
        return Dual(g, g.neg(self.v), {j: g.neg(n) for j, n in self.p.items()})

    def divc(self, c):   # Dual / Real
        g = self.g
        return Dual(g, g.div(self.v, c), {j: g.div(n, c) for j, n in self.p.items()})

    def addc(self, c):   # Dual + Real
        return Dual(self.g, self.g.add(self.v, c), dict(self.p))

    def mulc(self, c):   # Real * Dual
        g = self.g
        return Dual(g, g.mul(c, self.v), {j: g.mul(n, c) for j, n in self.p.items()})


class Dual2:
    """Second-order forward-mode number: value, gradient {j: node}, Hessian {(j, l), j <= l: node}.  Used for the
    Lagrangian Hessian (SURVEY.md 8f N3; no reference counterpart: src/moi.jl:26-28 offers [:Grad, :Jac] only)."""
    __slots__ = ("g", "v", "p", "h")

    def __init__(self, g, v, p=None, h=None):
        self.g = g
        self.v = v
        self.p = {j: n for j, n in (p or {}).items() if n != g.zero}
        self.h = {k: n for k, n in (h or {}).items() if n != g.zero}

    def part(self, j):
        return self.p.get(j, self.g.zero)

    def hess(self, j, l):
        return self.h.get((j, l) if j <= l else (l, j), self.g.zero)

    def _lin(self, o, op):
        g = self.g
        return Dual2(g, op(self.v, o.v), {j: op(self.part(j), o.part(j)) for j in sorted(set(self.p) | set(o.p))},
                     {k: op(self.h.get(k, g.zero), o.h.get(k, g.zero)) for k in sorted(set(self.h) | set(o.h))})

    def add(self, o):
        return self._lin(o, self.g.add)

    def sub(self, o):
        return self._lin(o, self.g.sub)

    def neg(self):
        g = self.g
        return Dual2(g, g.neg(self.v), {j: g.neg(n) for j, n in self.p.items()}, {k: g.neg(n) for k, n in self.h.items()})

    def mul(self, y):
        # (xy)' = y x' + x y';  (xy)'' = (y x'' + x y'') + (x'_j y'_l + x'_l y'_j)
        g, x = self.g, self
        p = {j: g.add(g.mul(y.v, x.part(j)), g.mul(x.v, y.part(j))) for j in sorted(set(x.p) | set(y.p))}
        keys = set(x.h) | set(y.h)
        for j in x.p:
            for l in y.p:
                keys.add((min(j, l), max(j, l)))
        h = {}
        for (j, l) in sorted(keys):
            t = g.add(g.mul(y.v, x.hess(j, l)), g.mul(x.v, y.hess(j, l)))
            c = g.add(g.mul(x.part(j), y.part(l)), g.mul(x.part(l), y.part(j)))
            h[(j, l)] = g.add(t, c)
        return Dual2(g, g.mul(x.v, y.v), p, h)

    def divc(self, c):
        g = self.g
        return Dual2(g, g.div(self.v, c), {j: g.div(n, c) for j, n in self.p.items()}, {k: g.div(n, c) for k, n in self.h.items()})

    def addc(self, c):
        return Dual2(self.g, self.g.add(self.v, c), dict(self.p), dict(self.h))

    def mulc(self, c):
        g = self.g
        return Dual2(g, g.mul(c, self.v), {j: g.mul(n, c) for j, n in self.p.items()}, {k: g.mul(n, c) for k, n in self.h.items()})


def contact_dynamics(g, mode, x, u, P):
    """planar_quadruped.jl:36-79 / :89-132 / :142-185 on Duals (x: 14, u: 5)."""
    zero = type(x[0])(g, g.zero)
    xb, yb = x[0], x[1]
    x1, y1 = x[3], x[4]
    x2, y2 = x[5], x[6]
    F1x, F1y, F2x, F2y = u[0], u[1], u[2], u[3]
    bax = F1x.add(F2x).divc(P["mb"])
    bay = F1y.add(F2y).divc(P["mb"]).addc(P["g"])
    t1 = F1x.neg().mul(y1.sub(yb))
    t2 = F1y.mul(x1.sub(xb))
    t3 = F2x.mul(y2.sub(yb))
    t4 = F2y.mul(x2.sub(xb))
    tau = t1.add(t2).sub(t3).add(t4)
    bw = tau.divc(P["Ib"])
    xd = [None] * 14
    xd[0], xd[1], xd[2] = x[7], x[8], x[9]
    xd[7], xd[8], xd[9] = bax, bay, bw
    if mode == 1:
        xd[3] = xd[4] = zero
        xd[5], xd[6] = x[12], x[13]
        xd[10] = xd[11] = zero
        xd[12] = F2x.neg().divc(P["mf"])
        xd[13] = F2y.neg().divc(P["mf"]).addc(P["g"])
    elif mode == 2:
        xd[3], xd[4] = x[10], x[11]
        xd[5] = xd[6] = zero
        xd[10] = F1x.neg().divc(P["mf"])
        xd[11] = F1y.neg().divc(P["mf"]).addc(P["g"])
        xd[12] = xd[13] = zero
    else:
        for i in (3, 4, 5, 6, 10, 11, 12, 13):
            xd[i] = zero
    return xd


def rk4(g, mode, x, u, P):
    """planar_quadruped.jl:189-221 on Duals (x: 15, u: 5)."""
    h = u[4]
    half, two, six = g.const(0.5), g.const(2.0), g.const(6.0)
    f1 = contact_dynamics(g, mode, x[:14], u, P)
    hh = h.mulc(half)
    f2 = contact_dynamics(g, mode, [x[i].add(hh.mul(f1[i])) for i in range(14)], u, P)
    f3 = contact_dynamics(g, mode, [x[i].add(hh.mul(f2[i])) for i in range(14)], u, P)
    f4 = contact_dynamics(g, mode, [x[i].add(h.mul(f3[i])) for i in range(14)], u, P)
    h6 = h.divc(six)
    xn = []
    for i in range(14):
        s = f1[i].add(f2[i].mulc(two)).add(f3[i].mulc(two)).add(f4[i])
        xn.append(x[i].add(h6.mul(s)))
    xn.append(x[14].add(u[4]))
    return xn


def build_hessian(mode):
    """lambda-contracted Hessian of one RK4 step: {(row, col), row >= col: node} with lam[i] as inputs."""
    g = Graph()
    P = {n: g.inp(n) for n in ("g", "mb", "mf", "Ib")}
    z = [Dual2(g, g.inp(f"x[{j}]" if j < NX else f"u[{j - NX}]"), {j: g.one}) for j in range(NP)]
    xn = rk4(g, mode, z[:NX], z[NX:], P)
    lam = [g.inp(f"lam[{i}]") for i in range(NX)]
    keys = set()
    for i in range(NX):
        keys |= set(xn[i].h)
    ent = {}
    for (j, l) in keys:                       # j <= l  ->  lower-triangle entry (row l, column j)
        acc = g.zero
        for i in range(NX):
            n = xn[i].h.get((j, l))
            if n is not None:
                acc = g.add(acc, g.mul(lam[i], n))
        ent[(l, j)] = acc
    return g, ent


def build(mode, with_partials):
    g = Graph()
    P = {n: g.inp(n) for n in ("g", "mb", "mf", "Ib")}
    z = []
    for j in range(NP):
        name = f"x[{j}]" if j < NX else f"u[{j - NX}]"
        z.append(Dual(g, g.inp(name), {j: g.one} if with_partials else None))
    xn = rk4(g, mode, z[:NX], z[NX:], P)
    return g, xn


# -------------------------------------------------------------------------------- emission
def emit_body(g, outputs, indent="    "):
    """outputs: list of (lhs_string, node).  Returns (lines, op_counts)."""
    live = set()
    stack = [n for _, n in outputs]
    while stack:
        n = stack.pop()
        if n in live:
            continue
        live.add(n)
        key = g.nodes[n]
        if key[0] in ("add", "sub", "mul", "div"):
            stack.extend(key[1:3])
        elif key[0] == "neg":
            stack.append(key[1])
    counts = {"add": 0, "sub": 0, "mul": 0, "div": 0, "neg": 0}

    def ref(n):
        key = g.nodes[n]
        if key[0] == "c":
            return repr(key[1])
        if key[0] == "in":
            return key[1] if "[" in key[1] else "K." + key[1]
        return f"t{n}"

    lines = []
    for n in sorted(live):
        key = g.nodes[n]
        op = key[0]
        if op in ("c", "in"):
            continue
        counts[op] += 1
        if op == "neg":
            lines.append(f"{indent}const double t{n} = -{ref(key[1])};")
        elif op == "div":
            # every divisor is a model constant (mb, mf, Ib) or the literal 6.0: name it, so the includer
            # can divide exactly with a precomputed reciprocal (QL_DIV_<name>(a) == RN(a / name))
            d = g.nodes[key[2]]
            name = {"mb": "MB", "mf": "MF", "Ib": "IB"}[d[1]] if d[0] == "in" else {6.0: "SIX"}[d[1]]
            lines.append(f"{indent}const double t{n} = QL_DIV_{name}({ref(key[1])});")
        else:
            mac = {"add": "QL_ADD", "sub": "QL_SUB", "mul": "QL_MUL"}[op]
            lines.append(f"{indent}const double t{n} = {mac}({ref(key[1])}, {ref(key[2])});")
    for lhs, n in outputs:
        lines.append(f"{indent}{lhs} = {ref(n)};")
    return lines, counts


def pattern_of(g, xn):
    """Column-major list of (i, j) whose partial is not structurally zero."""
    pat = []
    for j in range(NP):
        for i in range(NX):
            if xn[i].part(j) != g.zero:
                pat.append((i, j))
    return pat


# column groups of a knot's run (see layout.h): pointer index used by the patch code
def col_group(j):
    if j <= 1:
        return 0
    if j == 2:
        return 1
    if j <= 4:
        return 2
    if j <= 6:
        return 3
    if j <= 16:
        return 4
    if j <= 18:
        return 5
    return 6


def rk4_offset(i, j):
    """Offset (in doubles, before the group shift) of RK4-block entry (i, j) inside a knot's run."""
    if j < NX:
        return 30 * j + 15 + i
    return 450 + 15 * (j - NX) + i


def fold(terms):
    """Left fold of the terms with QL_ADD, starting from the first term."""
    expr = terms[0]
    for t in terms[1:]:
        expr = f"QL_ADD({expr}, {t})"
    return expr


def emit_products(w, mode, g, xn, pat, var, keep, union, hidx, obj):
    """Matrix-free products of one mode (matrix times vector, no matrix in memory).  Every output entry is the left
    fold of entry * vector terms over the structurally non-zero entries (the SPARSE_TRUE pattern / the Hessian's union
    pattern), in ascending column order for J w and the Hessian, ascending row order for J' y.  Structural constants
    are folded in: a +1 entry contributes the vector element itself, a -1 entry its negation (both exact)."""
    w = w.append
    vidx = {e: n for n, e in enumerate(var)}

    def term(i, j, vec):
        if (i, j) in vidx:
            return f"QL_MUL(jv[{vidx[(i, j)]}], {vec})"
        c = g.cval(xn[i].part(j))
        if c == 1.0:
            return vec
        if c == -1.0:
            return f"-{vec}"
        return f"QL_MUL({c!r}, {vec})"

    for jump in ((0, 1) if mode != 3 else (0,)):
        pj = [(i, j) for (i, j) in pat if not (jump and not keep[i])]
        fn = f"mode{mode}" + ("_jump" if jump else "")
        w(f"// J w for the 15 defect rows of a knot in {fn}: the RK4 block (jv + constants) times w = [x_k; u_k] in")
        w(f"// ascending column order, then the -I block times wn = x_(k+1) (a + (-b) is a - b bit for bit)")
        w(f"QL_FN void ql_rk4_jvp_{fn}(const double* jv, const double* w, const double* wn, double* out)")
        w("{")
        for i in range(NX):
            terms = [term(i, j, f"w[{j}]") for (ii, j) in sorted(pj, key=lambda e: e[1]) if ii == i]
            w(f"    out[{i}] = {f'QL_SUB({fold(terms)}, wn[{i}])' if terms else f'-wn[{i}]'};")
        w("}")
        w("")
        w(f"// J' y over the 20 columns of a knot's RK4 block in {fn}: y = the knot's 15 defect multipliers, rows in")
        w(f"// ascending order.  State column j continues the fold a[j] of the rows above the block (init / term / -I).")
        w(f"QL_FN void ql_rk4_vjp_{fn}(const double* jv, const double* y, const double* a, double* out)")
        w("{")
        for j in range(NP):
            terms = [term(i, j, f"y[{i}]") for (i, jj) in pj if jj == j]
            if j < NX:
                terms = [f"a[{j}]"] + terms
            assert terms, (fn, j)
            w(f"    out[{j}] = {fold(terms)};")
        w("}")
        w("")
    w(f"// Hessian block of a knot in mode {mode} times v (the knot's 20 variables): row i of the symmetric block in")
    w(f"// ascending column order; each entry formed exactly as ql_hess_store_mode{mode} forms it")
    w(f"QL_FN void ql_hess_prod_mode{mode}(const double* hv, const double* ox, const double* ou, const double* hx,")
    w(f"                                  const double* hu, double hh, double tt, const double* v, double* out)")
    w("{")
    pos_of = {}
    for pos, k in enumerate(union):
        terms = []
        if k in hidx:
            terms.append(f"hv[{hidx[k]}]")
        if k in obj:
            terms.append(obj[k])
        if k == (2, 2):
            terms.append("tt")
        w(f"    const double e{pos} = {fold(terms)};")
        pos_of[k] = pos
    for i in range(NP):
        terms = []
        for c in range(NP):
            k = (i, c) if c <= i else (c, i)
            if k in pos_of:
                terms.append(f"QL_MUL(e{pos_of[k]}, v[{c}])")
        w(f"    out[{i}] = {fold(terms)};")
    w("}")
    w("")


def main():
    out = []
    w = out.append
    w("// GENERATED by tools/gen_rk4_dual.py -- do not edit by hand.")
    w("//")
    w("// Straight-line fp64 code for one RK4 step of the hybrid planar-quadruped dynamics")
    w("// (reference: src/planar_quadruped.jl:36-221) and for the structurally non-zero entries")
    w("// of its 15x20 Jacobian w.r.t. [x;u] (reference: ForwardDiff.jacobian, :225-248).")
    w("// Operation order and operand pairing follow the reference / ForwardDiff 0.10.25 dual")
    w("// rules exactly; operations whose result is exact (x*0, x*1, x+0, ...) are removed, so")
    w("// the results are bit-identical to the dense 20-wide dual evaluation for finite inputs.")
    w("//")
    w("// The includer defines QL_ADD/QL_SUB/QL_MUL (round-to-nearest, NO fma contraction),")
    w("// QL_DIV_MB/QL_DIV_MF/QL_DIV_IB/QL_DIV_SIX(a) (correctly rounded a/mb, a/mf, a/Ib, a/6.0; they may use")
    w("// the constants object K, whose type KT also provides the fields K.g, K.mb, K.mf, K.Ib),")
    w("// QL_FN (function qualifiers) and QL_ST(ptr, off, val) (store of one double).")
    w("#pragma once")
    w("")
    summary = []
    prod = []           # the product routines go after everything else: the routines above stay as they were
    for mode in (1, 2, 3):
        # primal only
        g, xn = build(mode, False)
        lines, cnt = emit_body(g, [(f"xn[{i}]", xn[i].v) for i in range(NX)])
        w(f"// mode {mode}, values only: {cnt}")
        w(f"template <typename KT>")
        w(f"QL_FN void ql_rk4_mode{mode}(const double* x, const double* u, const KT& K, double* xn)")
        w("{")
        out.extend(lines)
        w("}")
        w("")
        summary.append((mode, "primal", cnt))
        # with partials
        g, xn = build(mode, True)
        pat = pattern_of(g, xn)
        var = [(i, j) for (i, j) in pat if not g.is_const(xn[i].part(j))]
        con = [(i, j) for (i, j) in pat if g.is_const(xn[i].part(j))]
        outs = [(f"xn[{i}]", xn[i].v) for i in range(NX)]
        outs += [(f"jv[{n}]", xn[i].part(j)) for n, (i, j) in enumerate(var)]
        lines, cnt = emit_body(g, outs)
        w(f"// mode {mode}, values + Jacobian: pattern of {len(pat)} entries = {len(var)} value-dependent (jv) + {len(con)} constants: {cnt}")
        w(f"#define QL_NJ_MODE{mode} {len(var)}")
        w(f"#define QL_NJC_MODE{mode} {len(con)}")
        w(f"template <typename KT>")
        w(f"QL_FN void ql_rk4_jac_mode{mode}(const double* x, const double* u, const KT& K, double* xn, double* jv)")
        w("{")
        out.extend(lines)
        w("}")
        w("")
        w(f"// value-dependent entries of mode {mode}: jv[n] = d xn[PAT_I[n]] / d z[PAT_J[n]], column-major order")
        w(f"static const unsigned char QL_PAT_I_MODE{mode}[{len(var)}] = {{{', '.join(str(i) for i, _ in var)}}};")
        w(f"static const unsigned char QL_PAT_J_MODE{mode}[{len(var)}] = {{{', '.join(str(j) for _, j in var)}}};")
        w(f"// constant entries of mode {mode} (value QL_CPAT_V)")
        w(f"static const unsigned char QL_CPAT_I_MODE{mode}[{len(con)}] = {{{', '.join(str(i) for i, _ in con)}}};")
        w(f"static const unsigned char QL_CPAT_J_MODE{mode}[{len(con)}] = {{{', '.join(str(j) for _, j in con)}}};")
        w(f"static const double QL_CPAT_V_MODE{mode}[{len(con)}] = {{{', '.join(repr(g.cval(xn[i].part(j))) for i, j in con)}}};")
        w("")
        keep = (1, 1, 1, 1, 0, 1, 0, 1, 1, 1, 0, 0, 0, 0, 0)
        w(f"// Patch the value-dependent entries into a knot's run.  p[grp] addresses the run start shifted by the")
        w(f"// extras that precede column group grp (layout.h: ql_col_group / ql_group_shift).  `jump` applies the")
        w(f"// reference's jump Jacobian Diagonal([1,1,1,1,0,1,0,1,1,1,0,0,0,0,0]) (planar_quadruped.jl:262-263).")
        w(f"template <typename PTR>")
        w(f"QL_FN void ql_patch_mode{mode}(const double* jv, const PTR* p, bool jump)")
        w("{")
        for n, (i, j) in enumerate(var):
            val = f"jv[{n}]" if keep[i] else f"(jump ? 0.0 : jv[{n}])"
            w(f"    QL_ST(p[{col_group(j)}], {rk4_offset(i, j)}, {val});")
        w("}")
        w("")
        w(f"// The constant entries (part of a staging buffer's persistent image; rewritten only on a rebuild).")
        w(f"template <typename PTR>")
        w(f"QL_FN void ql_const_mode{mode}(const PTR* p, bool jump)")
        w("{")
        for (i, j) in con:
            v = repr(g.cval(xn[i].part(j)))
            val = v if keep[i] else f"(jump ? 0.0 : {v})"
            w(f"    QL_ST(p[{col_group(j)}], {rk4_offset(i, j)}, {val});")
        w("}")
        w("")
        # ---- SPARSE_TRUE: only the structurally non-zero entries, identity blocks as diagonals ---------------
        # Run of a knot k < N in SPARSE_TRUE order: state column j = [diag entry] [pattern rows of column j]
        # [extras], control column j = [pattern rows] [final-ctrl extra].  Offsets below exclude the extras;
        # the group pointers p[grp] add them exactly as for SPARSE_BLOCK (same column groups).
        for jump in ((0, 1) if mode != 3 else (0,)):
            pj = [(i, j) for (i, j) in pat if not (jump and not keep[i])]
            npat = [sum(1 for (_, jj) in pj if jj == j) for j in range(NP)]
            base = []
            acc = 0
            for j in range(NP):
                base.append(acc)
                acc += (1 if j < NX else 0) + npat[j]
            tag = f"MODE{mode}" + ("_JUMP" if jump else "")
            fn = f"mode{mode}" + ("_jump" if jump else "")
            w(f"// SPARSE_TRUE, {tag}: {len(pj)} pattern entries; run length without extras = {acc}")
            w(f"#define QL_TRUE_NPAT_{tag} {len(pj)}")
            w(f"#define QL_TRUE_LEN_{tag} {acc}")
            w(f"// offset (without extras) just past column j's entries = where column j's extra row goes")
            w(f"static const unsigned short QL_TRUE_COLEND_{tag}[{NP}] = {{{', '.join(str(base[j] + (1 if j < NX else 0) + npat[j]) for j in range(NP))}}};")
            colend = [base[j] + (1 if j < NX else 0) + npat[j] for j in range(NP)]
            for j in (1, 2, 4, 6, 16, 18):
                w(f"#define QL_TRUE_X{j}_{tag} {colend[j]}")
            w(f"static const unsigned char QL_TRUE_I_{tag}[{len(pj)}] = {{{', '.join(str(i) for i, _ in pj)}}};")
            w(f"static const unsigned char QL_TRUE_J_{tag}[{len(pj)}] = {{{', '.join(str(j) for _, j in pj)}}};")
            w(f"// writes the 15 diagonal entries (value dg: +1 for the init block of knot 1, -1 otherwise) and every")
            w(f"// pattern entry of the RK4 block (jv = value-dependent entries, constants inline)")
            w(f"template <typename PTR>")
            w(f"QL_FN void ql_store_true_{fn}(const double* jv, const PTR* p, double dg)")
            w("{")
            for j in range(NX):
                w(f"    QL_ST(p[{col_group(j)}], {base[j]}, dg);")
            vidx = {e: n for n, e in enumerate(var)}
            for j in range(NP):
                r = 0
                for (i, jj) in pj:
                    if jj != j:
                        continue
                    off = base[j] + (1 if j < NX else 0) + r
                    r += 1
                    if (i, j) in vidx:
                        w(f"    QL_ST(p[{col_group(j)}], {off}, jv[{vidx[(i, j)]}]);")
                    else:
                        w(f"    QL_ST(p[{col_group(j)}], {off}, {repr(g.cval(xn[i].part(j)))});")
            w("}")
            w("")
        # ---- VALS: only the value-dependent entries (what a host caller with a registered, pre-filled row needs) ----
        # Run of a knot k < N: the jv entries in column-major order (masked rows dropped at the jump knot) with the
        # body-clearance d/dtheta entry (constraints.jl:269-273) at its column-major place: after column 2.
        for jump in ((0, 1) if mode != 3 else (0,)):
            vj = [(n, i, j) for n, (i, j) in enumerate(var) if not (jump and not keep[i])]
            tag = f"MODE{mode}" + ("_JUMP" if jump else "")
            fn = f"mode{mode}" + ("_jump" if jump else "")
            w(f"// VALS, {tag}: {len(vj)} value-dependent RK4 entries + d/dtheta")
            w(f"#define QL_VALS_LEN_{tag} {len(vj) + 1}")
            w(f"template <typename PTR>")
            w(f"QL_FN void ql_store_vals_{fn}(const double* jv, double jtheta, PTR run)")
            w("{")
            pos, theta_done = 0, False
            for n, i, j in vj:
                if j >= 3 and not theta_done:
                    w(f"    QL_ST(run, {pos}, jtheta);")
                    pos += 1
                    theta_done = True
                w(f"    QL_ST(run, {pos}, jv[{n}]);")
                pos += 1
            assert theta_done and pos == len(vj) + 1
            w("}")
            w("")
        summary.append((mode, "jac", cnt, len(var), len(con)))
        # ---- Lagrangian Hessian block of a knot (N3): sum_i lam_i Hess(rk4_i) + sigma Hess(h * stagecost) + the
        # body-clearance row's d2/dtheta2, lower triangle of the 20x20 block in column-major order -----------------
        gh, ent = build_hessian(mode)
        hkeys = sorted(ent, key=lambda rc: (rc[1], rc[0]))             # by (column, row)
        lines, cnt = emit_body(gh, [(f"hv[{n}]", ent[k]) for n, k in enumerate(hkeys)])
        w(f"// mode {mode}, lambda-contracted Hessian of the RK4 step: {len(hkeys)} entries of the lower triangle: {cnt}")
        w(f"#define QL_NH_MODE{mode} {len(hkeys)}")
        w(f"template <typename KT>")
        w(f"QL_FN void ql_rk4_hess_mode{mode}(const double* x, const double* u, const KT& K, const double* lam, double* hv)")
        w("{")
        out.extend(lines)
        w("}")
        w("")
        # objective: f_k = h * stagecost(x, u) (costs.jl:12): d2/dx_i2 = h Q_ii, d2/du_i2 = h R_ii (i < 4),
        # d2/dh dx_i = (Qx+q)_i, d2/dh du_i = (Ru+r)_i, d2/dh2 = 2 (R_55 h + r_5) + h R_55; all times sigma
        obj = {(i, i): f"ox[{i}]" for i in range(NX)}
        obj.update({(NX + i, NX + i): f"ou[{i}]" for i in range(NU - 1)})
        obj.update({(NP - 1, i): f"hx[{i}]" for i in range(NX)})
        obj.update({(NP - 1, NX + i): f"hu[{i}]" for i in range(NU - 1)})
        obj[(NP - 1, NP - 1)] = "hh"
        union = sorted(set(hkeys) | set(obj) | {(2, 2)}, key=lambda rc: (rc[1], rc[0]))
        hidx = {k: n for n, k in enumerate(hkeys)}
        w(f"// union pattern of a knot's Hessian block in mode {mode}: {len(union)} entries (row, col), row >= col, column-major")
        w(f"#define QL_HESS_LEN_MODE{mode} {len(union)}")
        w(f"static const unsigned char QL_HESS_R_MODE{mode}[{len(union)}] = {{{', '.join(str(r) for r, _ in union)}}};")
        w(f"static const unsigned char QL_HESS_C_MODE{mode}[{len(union)}] = {{{', '.join(str(c) for _, c in union)}}};")
        w(f"// writes the block: RK4 part (hv) + objective part (ox, ou, hx, hu, hh: already scaled by sigma) + tt on (theta, theta)")
        w(f"template <typename PTR>")
        w(f"QL_FN void ql_hess_store_mode{mode}(const double* hv, const double* ox, const double* ou, const double* hx,")
        w(f"                                   const double* hu, double hh, double tt, PTR run)")
        w("{")
        for pos, k in enumerate(union):
            terms = []
            if k in hidx:
                terms.append(f"hv[{hidx[k]}]")
            if k in obj:
                terms.append(obj[k])
            if k == (2, 2):
                terms.append("tt")
            expr = terms[0]
            for t in terms[1:]:
                expr = f"QL_ADD({expr}, {t})"
            w(f"    QL_ST(run, {pos}, {expr});")
        w("}")
        w("")
        summary.append((mode, "hess", cnt, len(hkeys), len(union)))
        emit_products(prod, mode, g, xn, pat, var, keep, union, hidx, obj)
    out.extend(prod)
    text = "\n".join(out) + "\n"
    with open(OUT, "w") as f:
        f.write(text)
    for s in summary:
        print(s, file=sys.stderr)
    print("wrote", os.path.normpath(OUT), file=sys.stderr)


if __name__ == "__main__":
    main()
