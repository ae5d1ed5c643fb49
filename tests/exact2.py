"""Exact reference for programs with two decision variables, in rational arithmetic.

    minimise  1/2 z'Pz + q'z + sum_i w_i |a_i z - kink_i|   subject to  l <= Az <= u,   z in R^2

Every float64 input is converted to a `fractions.Fraction` exactly, so the optimum below is the optimum of the program
the floats describe, with no rounding and no tolerance.  The minimiser is found by enumeration:

  * every intersection of two non-parallel lines, where the lines are the finite bounds a_i z = l_i, a_i z = u_i and
    the kinks a_i z = kink_i of the |.| rows;
  * on each line, between consecutive breakpoints (its intersections with the other lines), the minimiser of the
    quadratic that holds on that piece -- the sides of the |.| rows are read at a point inside the piece;
  * for P positive definite, the stationary point of every sign pattern of the |.| rows.

Every candidate is checked for feasibility exactly and the cost is evaluated exactly there.  Whatever the objective, a
minimiser over a bounded polygon lies in one of these sets, so the smallest cost among the feasible candidates is the
optimum.  Boundedness is asserted, not assumed.

Plain and slow on purpose: it shares no code with oracle/qp.py or with the active-set logic of the kernels.
"""
from __future__ import annotations

from dataclasses import dataclass
from fractions import Fraction
from itertools import combinations, product
from typing import List, Optional, Tuple

import numpy as np

F0 = Fraction(0)


def fr(x) -> Optional[Fraction]:
    """float64 -> Fraction, exactly; +-inf -> None (no bound)."""
    x = float(x)
    if np.isnan(x):
        raise ValueError("NaN in a program")
    return None if np.isinf(x) else Fraction(x)


@dataclass
class Result:
    feasible: bool
    f: Optional[Fraction]                   # optimum (None when infeasible)
    argmin: List[Tuple[Fraction, Fraction]]  # the optimal candidates (distinct points)
    lines: list                             # (a0, a1, c) of every line used, for the active sets of `active_rows`

    @property
    def status(self) -> int:
        return 0 if self.feasible else 2

    @property
    def v0_unique(self) -> bool:
        return self.feasible and len({z[0] for z in self.argmin}) == 1


def _dot(a, z):
    return a[0] * z[0] + a[1] * z[1]


def _objective(P, q, absr, z):
    f = (P[0][0] * z[0] * z[0] + 2 * P[0][1] * z[0] * z[1] + P[1][1] * z[1] * z[1]) / 2 + q[0] * z[0] + q[1] * z[1]
    for a, k, w in absr:
        f += w * abs(_dot(a, z) - k)
    return f


def _feasible(rows, z) -> bool:
    for a, lo, hi in rows:
        t = _dot(a, z)
        if (lo is not None and t < lo) or (hi is not None and t > hi):
            return False
    return True


def _perp(a):
    return (-a[1], a[0])


def _bounded(rows) -> bool:
    """The polygon {z: l <= Az <= u} (non-empty) is bounded iff its recession cone {d: a_i d <= 0 where u_i is finite,
    a_i d >= 0 where l_i is finite} is {0}.  A non-zero closed cone in the plane contains a direction orthogonal to one
    of the constraining rows (an extreme ray, the boundary of a half-plane, or the line it contains), so only those
    directions need testing."""
    cons = [(a, lo, hi) for a, lo, hi in rows if (a[0] or a[1]) and (lo is not None or hi is not None)]
    if not cons:
        return False
    for a, _, _ in cons:
        for s in (1, -1):
            d = (s * _perp(a)[0], s * _perp(a)[1])
            if all((hi is None or _dot(b, d) <= 0) and (lo is None or _dot(b, d) >= 0) for b, lo, hi in cons):
                return False
    return True


def exact_qp2(P, q, A, l, u, kink=None, wabs=None) -> Result:
    """P (2, 2) symmetric positive semidefinite, q (2,), A (m, 2), l / u (m,) with +-inf for a missing bound,
    kink / wabs (m,): row i adds wabs_i |a_i z - kink_i| to the cost when wabs_i > 0.  Float arrays or Fractions."""
    m = len(A)
    kink = np.zeros(m) if kink is None else kink
    wabs = np.zeros(m) if wabs is None else wabs
    cv = lambda x: x if (x is None or isinstance(x, Fraction)) else fr(x)          # noqa: E731
    P = [[cv(P[i][j]) for j in range(2)] for i in range(2)]
    assert P[0][1] == P[1][0], "P must be symmetric"
    q = [cv(q[0]), cv(q[1])]
    rows, absr = [], []
    for i in range(m):
        a = (cv(A[i][0]), cv(A[i][1]))
        lo, hi = cv(l[i]), cv(u[i])
        rows.append((a, lo, hi))
        w = cv(wabs[i])
        if w and w > 0:
            absr.append((a, cv(kink[i]), w))
    # rows with a = 0 are constants: feasible or not, whatever z is
    for a, lo, hi in rows:
        if not (a[0] or a[1]) and ((lo is not None and lo > 0) or (hi is not None and hi < 0)):
            return Result(False, None, [], [])
    lines, seen = [], set()                       # a z = c, normalised so that the first non-zero entry of a is 1
    for a, c in [(a, lo) for a, lo, _ in rows] + [(a, hi) for a, _, hi in rows] + [(a, k) for a, k, _ in absr]:
        if c is None or not (a[0] or a[1]):
            continue
        s = a[0] if a[0] else a[1]
        key = (a[0] / s, a[1] / s, c / s)
        if key not in seen:
            seen.add(key)
            lines.append(key)
    # ---- feasibility: with two independent constraining rows a non-empty polygon has a vertex; with fewer it contains
    # a line, so it is unbounded if it is not empty
    cand = set()
    for (a0, a1, c), (b0, b1, d) in combinations(lines, 2):
        det = a0 * b1 - a1 * b0
        if det:
            cand.add(((c * b1 - d * a1) / det, (a0 * d - b0 * c) / det))
    bound_lines = {(a[0] / (a[0] or a[1]), a[1] / (a[0] or a[1])) for a, lo, hi in rows
                   if (a[0] or a[1]) and (lo is not None or hi is not None)}
    has_vertex = any(x[0] * y[1] - x[1] * y[0] for x, y in combinations(bound_lines, 2))
    if has_vertex:
        if not any(_feasible(rows, z) for z in cand):
            return Result(False, None, [], lines)
    else:
        # all constraining rows parallel to one direction ref: an interval condition on t = ref z
        if not bound_lines:
            raise AssertionError("the feasible set is not bounded")
        ref = next(iter(bound_lines))
        lo_t, hi_t = None, None
        for a, lo, hi in rows:
            if not (a[0] or a[1]) or (lo is None and hi is None):
                continue
            s = a[0] / ref[0] if ref[0] else a[1] / ref[1]          # a = s * ref
            los, his = (lo, hi) if s > 0 else (hi, lo)
            if los is not None:
                lo_t = los / s if lo_t is None else max(lo_t, los / s)
            if his is not None:
                hi_t = his / s if hi_t is None else min(hi_t, his / s)
        if lo_t is not None and hi_t is not None and lo_t > hi_t:
            return Result(False, None, [], lines)
        raise AssertionError("the feasible set is not bounded")
    assert _bounded(rows), "the feasible set is not bounded"
    # ---- on each line: breakpoints and the minimiser of each piece
    for (a0, a1, c) in lines:
        n2 = a0 * a0 + a1 * a1
        z0 = (a0 * c / n2, a1 * c / n2)
        d = (-a1, a0)
        ts = set()
        for (b0, b1, e) in lines:
            bd = b0 * d[0] + b1 * d[1]
            if bd:
                ts.add((e - (b0 * z0[0] + b1 * z0[1])) / bd)
        ts = sorted(ts)
        if ts:
            probes = [ts[0] - 1] + [(x + y) / 2 for x, y in zip(ts, ts[1:])] + [ts[-1] + 1]
            ends = [(None, ts[0])] + list(zip(ts, ts[1:])) + [(ts[-1], None)]
        else:
            probes, ends = [F0], [(None, None)]
        Pd = (P[0][0] * d[0] + P[0][1] * d[1], P[1][0] * d[0] + P[1][1] * d[1])
        curv = d[0] * Pd[0] + d[1] * Pd[1]
        if curv <= 0:
            continue                              # linear along the line: its minimum over a piece is at a breakpoint
        for tp, (t_lo, t_hi) in zip(probes, ends):
            zp = (z0[0] + tp * d[0], z0[1] + tp * d[1])
            g = [P[0][0] * z0[0] + P[0][1] * z0[1] + q[0], P[1][0] * z0[0] + P[1][1] * z0[1] + q[1]]
            for a, k, w in absr:
                r = _dot(a, zp) - k
                if r:
                    sg = w if r > 0 else -w
                    g[0] += sg * a[0]
                    g[1] += sg * a[1]
            t = -(d[0] * g[0] + d[1] * g[1]) / curv
            if (t_lo is None or t >= t_lo) and (t_hi is None or t <= t_hi):
                cand.add((z0[0] + t * d[0], z0[1] + t * d[1]))
    # ---- P positive definite: the stationary point of every sign pattern of the |.| rows
    det = P[0][0] * P[1][1] - P[0][1] * P[1][0]
    if P[0][0] > 0 and det > 0:
        for signs in product((1, -1), repeat=len(absr)):
            g = list(q)
            for s, (a, _, w) in zip(signs, absr):
                g[0] += s * w * a[0]
                g[1] += s * w * a[1]
            cand.add((-(P[1][1] * g[0] - P[0][1] * g[1]) / det, -(P[0][0] * g[1] - P[1][0] * g[0]) / det))
    best, arg = None, []
    for z in cand:
        if not _feasible(rows, z):
            continue
        f = _objective(P, q, absr, z)
        if best is None or f < best:
            best, arg = f, [z]
        elif f == best:
            arg.append(z)
    assert best is not None
    return Result(True, best, sorted(arg), lines)


def active_rows(prog_rows, z) -> frozenset:
    """Rows (index, side) that hold with equality at z: side 'l', 'u' or 'k' (on the kink).  `prog_rows` as returned
    by `Instance.rows`."""
    out = set()
    for i, (a, lo, hi, k, w) in enumerate(prog_rows):
        t = _dot(a, z)
        if lo is not None and t == lo:
            out.add((i, "l"))
        if hi is not None and t == hi:
            out.add((i, "u"))
        if w and t == k:
            out.add((i, "k"))
    return frozenset(out)


@dataclass
class Instance:
    """A CompiledProgram evaluated at one parameter point, exactly."""
    P: list
    q: list
    A: list
    l: list
    u: list
    kink: list
    wabs: list
    c0: Fraction            # cost constant: the program's cost is the QP's plus c0
    chk_ok: bool            # every parametric feasibility row Rchk [1; p; alpha] <= 0

    @property
    def rows(self):
        return [(self.A[i], self.l[i], self.u[i], self.kink[i], self.wabs[i]) for i in range(len(self.A))]

    def solve(self) -> Result:
        if not self.chk_ok:
            return Result(False, None, [], [])
        r = exact_qp2(self.P, self.q, self.A, self.l, self.u, self.kink, self.wabs)
        if r.feasible:
            r.f = r.f + self.c0
        return r


def _matvec(M, x):
    return [sum((fr(M[i][j]) * x[j] for j in range(len(x)) if M[i][j] != 0.0), F0) for i in range(len(M))]


def at_point(prog, xbar0, e0) -> Instance:
    """The CompiledProgram `prog` (tzddpc_b200/program.py) at p = [xbar0; e0]: r = R [1; p; |Bt p + gam|], bounds
    l0 + r / u0 + r, kinks kink0 + r, q = q0 + Qp p, cost constant cc [1; p; alpha] + p' CC2 p -- the reading of
    tests/common.py:solve_compiled, in exact arithmetic."""
    assert prog.nz == 2, "the exact reference is for two decision variables"
    p = [fr(x) for x in np.r_[xbar0, e0]]
    alpha = [abs(s + fr(g)) for s, g in zip(_matvec(prog.Bt, p), prog.gam)] if prog.na else []
    w = [Fraction(1)] + p + alpha
    chk_ok = all(s <= 0 for s in _matvec(prog.Rchk, w)) if prog.Rchk.shape[0] else True
    r = _matvec(prog.R, w)
    add = lambda b, s: None if np.isinf(b) else fr(b) + s                                     # noqa: E731
    l = [add(prog.l0[i], r[i]) for i in range(prog.nc)]
    u = [add(prog.u0[i], r[i]) for i in range(prog.nc)]
    kink = [fr(prog.kink0[i]) + r[i] if prog.wabs[i] > 0 else F0 for i in range(prog.nc)]
    wabs = [fr(x) for x in prog.wabs]
    qp = _matvec(prog.Qp, p)
    q = [fr(prog.q0[j]) + qp[j] for j in range(2)]
    c2 = _matvec(prog.CC2, p)
    c0 = sum((fr(c) * x for c, x in zip(prog.cc, w) if c != 0.0), F0) + sum((a * b for a, b in zip(p, c2)), F0)
    A = [(fr(prog.A[i][0]), fr(prog.A[i][1])) for i in range(prog.nc)]
    P = [[fr(prog.P[i][j]) for j in range(2)] for i in range(2)]
    return Instance(P, q, A, l, u, kink, wabs, c0, chk_ok)


def solve_at(prog, xbar0, e0) -> Result:
    return at_point(prog, xbar0, e0).solve()


def cost_at(inst: Instance, z) -> Fraction:
    """The program's cost at z (the QP objective plus c0), feasible or not."""
    absr = [(inst.A[i], inst.kink[i], inst.wabs[i]) for i in range(len(inst.A)) if inst.wabs[i] > 0]
    return _objective(inst.P, inst.q, absr, [fr(z[0]) if not isinstance(z[0], Fraction) else z[0],
                                             fr(z[1]) if not isinstance(z[1], Fraction) else z[1]]) + inst.c0
