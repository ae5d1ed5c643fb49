"""The exact two-variable reference (tests/exact2.py) on hand-built programs with known answers, and against the
interior-point reading of the shipped examples' compiled programs (tests/common.py:solve_compiled)."""
from fractions import Fraction as Fr

import numpy as np
import pytest

from tests import common, exact2
from tzddpc_b200 import configs

INF = np.inf


def _qp(P, q, rows, kinks=None):
    """rows: (a0, a1, lo, hi); kinks: {row: (kink, w)}"""
    A = np.array([r[:2] for r in rows], dtype=float)
    lo = np.array([r[2] for r in rows], dtype=float)
    hi = np.array([r[3] for r in rows], dtype=float)
    kink, wabs = np.zeros(len(rows)), np.zeros(len(rows))
    for i, (k, w) in (kinks or {}).items():
        kink[i], wabs[i] = k, w
    return exact2.exact_qp2(np.asarray(P, dtype=float), np.asarray(q, dtype=float), A, lo, hi, kink, wabs)


def test_unique_vertex():
    r = _qp(np.eye(2), [-3, -3], [(1, 0, -10, 1), (0, 1, -10, 1)])
    assert r.feasible and r.f == -5 and r.argmin == [(1, 1)] and r.v0_unique


def test_three_rows_through_one_vertex():
    r = _qp(np.zeros((2, 2)), [1, 1], [(1, 0, 0, 1), (0, 1, 0, 1), (1, 1, 0, INF)])
    assert r.feasible and r.f == 0 and r.argmin == [(0, 0)]


def test_lp_with_an_optimal_edge():
    r = _qp(np.zeros((2, 2)), [0, 1], [(1, 0, 0, 1), (0, 1, 0, 1)])
    assert r.feasible and r.f == 0
    assert (0, 0) in r.argmin and (1, 0) in r.argmin and all(z[1] == 0 for z in r.argmin)
    assert not r.v0_unique


def test_parallel_rows_one_an_equality():
    r = _qp(np.eye(2), [0, 0], [(1, 1, 1, 1), (1, 1, -INF, 2), (1, 0, -5, 5)])
    assert r.feasible and r.f == Fr(1, 4) and r.argmin == [(Fr(1, 2), Fr(1, 2))]


def test_kink_row_resting_on_a_bound_below_its_kink():
    # |z0 - 1| + z1^2 / 2 with z0 <= 0.6 on the same row: the row sits on its bound, on the lower side of its kink
    r = _qp([[0, 0], [0, 1]], [0, 0], [(1, 0, -3, 0.6), (0, 1, -1, 1)], {0: (1.0, 1.0)})
    assert r.feasible and r.f == 1 - Fr(0.6) and r.argmin == [(Fr(0.6), 0)]


def test_kink_row_resting_exactly_on_its_kink():
    r = _qp([[0, 0], [0, 1]], [0.25, 0], [(1, 0, -3, 0.5), (0, 1, -1, 1)], {0: (0.5, 2.0)})
    assert r.feasible and r.f == Fr(1, 8) and r.argmin == [(Fr(1, 2), 0)]


def test_infeasible_pair_of_singleton_bounds():
    r = _qp(np.eye(2), [0, 0], [(1, 0, 1, INF), (2, 0, -INF, 1)])          # z0 >= 1 and 2 z0 <= 1, z1 free
    assert not r.feasible and r.status == 2
    r = _qp(np.eye(2), [0, 0], [(1, 0, 1, INF), (2, 0, -INF, 1), (0, 1, -1, 1)])
    assert not r.feasible


def test_rank_one_P():
    # (z0 + z1)^2 / 2 - (z0 + z1) on the box [-1, 1]^2: the optimal set is the segment z0 + z1 = 1 through the interior
    r = _qp([[1, 1], [1, 1]], [-1, -1], [(1, 0, -1, 1), (0, 1, -1, 1)])
    assert r.feasible and r.f == Fr(-1, 2)
    assert (0, 1) in r.argmin and (1, 0) in r.argmin and not r.v0_unique
    # a linear term that breaks the tie: unique minimiser on the boundary
    r = _qp([[1, 1], [1, 1]], [-2, 0], [(1, 0, -1, 1), (0, 1, -1, 1)])
    assert r.feasible and r.f == -2 and r.argmin == [(1, -1)]


def test_unbounded_polygon_is_refused():
    with pytest.raises(AssertionError, match="not bounded"):
        _qp(np.eye(2), [0, 0], [(1, 0, 0, 1)])
    with pytest.raises(AssertionError, match="not bounded"):
        _qp(np.eye(2), [0, 0], [(1, 0, 0, INF), (0, 1, 0, INF)])


# ---- the shipped examples' compiled programs ------------------------------------------------------------------------

def pulley_with_box():
    """The pulley with x_hi[0] = 0.6: its |.| cost row and the box row merge (test_gpu_hot_path.py's
    test_kink_row_resting_on_a_bound_away_from_its_kink)."""
    cfg = configs.pulley()
    hi = np.full(cfg.n, np.inf)
    hi[0] = 0.6
    cfg.box = dict(x_hi=hi)
    return cfg


PROGRAMS = ("double_integrator", "pulley", "fivedim", "pulley_box")


def config(name):
    return pulley_with_box() if name == "pulley_box" else configs.CONFIGS[name]()


def compiled(name):
    cfg = config(name)
    u, x = common.dataset(cfg)
    o, K = common.make_oracle(cfg, u, x)
    return cfg, o, common.make_compiled(cfg, o)


def sample_points(cfg, o, rng, count):
    """Alternately a point of test_gpu_parity._points (anywhere in X, |e| <= 0.4: many are infeasible) and a point
    near the example's x0 (within a tenth of X's width, |e| <= 0.1: most are feasible)."""
    Xi = o.zonotopes.X.interval
    x0, width = np.asarray(cfg.X0[0], dtype=np.float64), Xi.right_limit - Xi.left_limit
    pts = []
    while len(pts) < count:
        if len(pts) % 2:
            pts.append((Xi.left_limit + width * rng.uniform(0.05, 0.95, cfg.n), rng.uniform(-0.4, 0.4, cfg.n)))
        else:
            pts.append((x0 + 0.1 * width * rng.uniform(-1, 1, cfg.n), rng.uniform(-0.1, 0.1, cfg.n)))
    return pts


@pytest.mark.parametrize("name", PROGRAMS)
def test_examples_match_the_interior_point_reading(name):
    cfg, o, prog = compiled(name)
    rng = np.random.default_rng(17)
    pts = [(np.asarray(cfg.X0[0], dtype=np.float64), np.zeros(cfg.n))] + sample_points(cfg, o, rng, 19)
    n_ok = 0
    for xb, e in pts:
        r = exact2.solve_at(prog, xb, e)
        s = common.solve_compiled(prog, xb, e)
        assert r.status == s["status"], (xb, e, r.status, s["status"])
        if r.feasible:
            n_ok += 1
            f = float(r.f)
            assert abs(f - s["cost"]) <= 1e-7 * max(1.0, abs(f)), (xb, e, f, s["cost"])
            if r.v0_unique:
                assert abs(float(r.argmin[0][0]) - s["v"][0, 0]) <= 1e-6 * max(1.0, abs(float(r.argmin[0][0])))
    assert n_ok >= 5


def test_planted_pulley_vertex_is_feasible_and_not_optimal():
    """A vertex a hint can name without being optimal: rows 4 (1.044 v0 >= -0.9) and 20 (0.163 v0 + v1 >= -1.998) of the
    pulley's compiled program on their lower bounds, at x0 with e = 0.  The point is exactly feasible and costs more than
    the optimum by more than 1, so a certificate that accepts it is wrong by O(1)."""
    cfg, o, prog = compiled("pulley")
    x0, e0 = np.asarray(cfg.X0[0], dtype=np.float64), np.zeros(cfg.n)
    inst = exact2.at_point(prog, x0, e0)
    assert inst.l[4] is not None and inst.u[4] is None and inst.l[20] is not None and inst.u[20] is None
    (a0, a1), (b0, b1) = inst.A[4], inst.A[20]
    det = a0 * b1 - a1 * b0
    z = ((inst.l[4] * b1 - inst.l[20] * a1) / det, (a0 * inst.l[20] - b0 * inst.l[4]) / det)
    assert all((lo is None or a[0] * z[0] + a[1] * z[1] >= lo) and (hi is None or a[0] * z[0] + a[1] * z[1] <= hi)
               for a, lo, hi, _, _ in inst.rows)
    best = inst.solve()
    cost = exact2.cost_at(inst, z)
    assert best.feasible and cost - best.f > 1
    assert abs(float(best.f) - 1.0) < 1e-12 and abs(float(cost) - 2.8638) < 1e-4
