"""The references at two to four inputs, horizon one and up to four noise generators (CPU), so that they are trusted before
tests/test_gpu_input_dims.py compares the CUDA kernels with them.

* `random_config(n, m, N, gW, seed)`: the random systems of those tests.
* `evaluate_program`: the oracle's program evaluated at a given v (objective, largest scaled constraint violation), the
  certificate a kernel's v is checked with where v itself is not unique (quirk Q7 of oracle/program.py: the stage cost sees
  xbar_0 .. xbar_(N-1) only, so v_(N-1) enters only the constraints and horizon 1 is a pure feasibility problem).
* The host canonicaliser builds the program shapes the GPU tests rely on.
* oracle/gain.py at m > 1, gW > 2 and n = 1 .. 8, and on an unstabilisable pair.
"""
import numpy as np
import pytest

import oracle
from oracle import gain
from tests import common
from tzddpc_b200 import configs

# (n, m, N, gW) -> (nv, nz, nc) of the host canonicaliser's program
SHAPES = {(3, 2, 1, 1): (2, 2, 3), (5, 2, 1, 1): (2, 2, 3), (4, 3, 2, 1): (6, 9, 26), (6, 3, 2, 3): (6, 9, 30),
          (8, 4, 2, 1): (8, 12, 39), (7, 2, 2, 2): None, (4, 4, 3, 1): (12, 16, 49), (3, 4, 4, 1): (16, 27, 75),
          (2, 4, 4, 4): (16, 26, 67)}


def random_config(n, m, N, gW, seed, T=None):
    """A stable random plant with m distinct input columns, gW noise generators of distinct directions, Q > 0 on the states,
    an |.| term on state 0 and a user box on one state."""
    rng = np.random.default_rng(seed)
    A = rng.normal(size=(n, n))
    A *= 0.9 / max(np.abs(np.linalg.eigvals(A)).max(), 1e-9)
    B = rng.normal(size=(n, m)) * (1.0 + 0.25 * np.arange(m))          # distinct column norms: a permutation shows
    GW = rng.normal(size=(n, gW))
    GW *= 0.02 / np.abs(GW).max(axis=0)
    w = np.zeros(n); w[0] = 2.0
    r = rng.uniform(-0.5, 0.5, n)
    lo = np.full(n, -np.inf); hi = np.full(n, np.inf)
    j = 1 if n >= 2 else 0
    lo[j], hi[j] = -3.0, 3.0
    return configs.ExampleConfig(f"random{n}x{m}N{N}g{gW}", A, B, X0=(np.zeros(n), np.zeros((n, 1))), U=(np.zeros(m), 2.0 * np.eye(m)),
                                 W=(np.zeros(n), GW), X=(np.zeros(n), 4.0 * np.eye(n)), T=T or 60 + 20 * n,
                                 horizon=N, steps=10, cost=dict(Q=0.5 * np.eye(n), w_abs=w, x_ref=r),
                                 box=dict(x_lo=lo, x_hi=hi), noise="sample", seed=seed)


def shape_seed(n, m, N, gW):
    # (3, 4, 4, 1): the default seed's system sends the oracle's interior-point solver to its iteration limit (seconds a solve)
    return {(3, 4, 4, 1): 7}.get((n, m, N, gW), 1000 * n + 100 * m + 10 * N + gW)


def evaluate_program(o, xbar0, e0, v):
    """The oracle's program (OracleTZDDPC._assemble) at the decision v (N x m), each |.| epigraph variable at its least
    feasible value.  Returns (objective, largest constraint violation scaled by max(1, |rhs|)); the violation is infinite when
    the parameters alone violate a constraint."""
    P, q, c0, G, h, param_ok = o._assemble(np.asarray(xbar0, dtype=np.float64), np.asarray(e0, dtype=np.float64))
    v = np.asarray(v, dtype=np.float64).reshape(-1)
    nv, nt = v.size, P.shape[0] - v.size
    r0 = G.shape[0] - 2 * nt
    # atom i: rows r0 + 2i (a v - t <= -c) and r0 + 2i + 1 (-a v - t <= c), so its least t is max of the two left sides
    lhs = G[r0:, :nv] @ v - h[r0:]
    t = np.maximum(lhs[0::2], lhs[1::2])
    y = np.r_[v, t]
    obj = float(0.5 * y @ P @ y + q @ y + c0)
    viol = float(np.max(np.r_[0.0, (G @ y - h) / np.maximum(1.0, np.abs(h))])) if param_ok else np.inf
    return obj, viol


def build(cfg):
    u, x = common.dataset(cfg)
    o, K = common.make_oracle(cfg, u, x)
    return o, K, u, x


def sample_points(cfg, S, seed):
    """S points (xbar0, e0): the first half inside the state box, the second half reaching past X and the user box, so that
    some are infeasible and some lie near the boundary of feasibility."""
    rng = np.random.default_rng(seed)
    n = cfg.n
    h = S // 2
    xb = np.vstack([rng.uniform(-1.0, 1.0, size=(h, n)), rng.uniform(-4.2, 4.2, size=(S - h, n))])
    e = rng.uniform(-0.05, 0.05, size=(S, n))
    return xb, e


@pytest.mark.parametrize("shape", list(SHAPES))
def test_shapes_of_the_canonicalised_program(shape):
    n, m, N, gW = shape
    cfg = random_config(n, m, N, gW, shape_seed(*shape))
    assert len({tuple(c) for c in np.round(cfg.B.T, 12)}) == m
    o, K, _, _ = build(cfg)
    prog = common.make_compiled(cfg, o)
    assert (prog.n, prog.m, prog.N) == (n, m, N)
    if SHAPES[shape] is not None:
        assert (prog.nv, prog.nz, prog.nc) == SHAPES[shape]


@pytest.mark.parametrize("shape", list(SHAPES))
def test_certificate_helper_returns_the_oracles_optimum(shape):
    n, m, N, gW = shape
    cfg = random_config(n, m, N, gW, shape_seed(*shape))
    o, K, _, _ = build(cfg)
    xb, e = sample_points(cfg, 8, 7)
    feasible = 0
    for i in range(len(xb)):
        r = o.solve_status(xb[i], e[i])
        if r.status != 0:
            continue
        feasible += 1
        obj, viol = evaluate_program(o, xb[i], e[i], r.v)
        assert viol <= 1e-12, (i, viol)                       # zero up to the rounding of G y - h
        # the interior point keeps every epigraph variable a hair above its |.| (up to ~4e-7 relative at horizon 4): the
        # helper, which puts them at |.|, can only be lower
        assert obj <= r.cost + 1e-12 * abs(r.cost)
        assert common.cost_close(obj, r.cost, 0.0), (i, obj, r.cost)
        # a v that leaves the feasible set is seen as such: move v far along every input
        _, viol_far = evaluate_program(o, xb[i], e[i], r.v + 50.0)
        assert viol_far > 1e-3
    assert feasible >= 2, f"{shape}: too few feasible points"


def _wz(n, gW, seed):
    rng = np.random.default_rng(seed)
    GW = rng.normal(size=(n, gW)) * 0.02
    return np.hstack([np.zeros((n, 1)), GW])


@pytest.mark.parametrize("n,m", [(1, 2), (3, 3), (7, 4), (8, 2)])
def test_oracle_lqr_gain_matches_scipy_at_several_inputs(n, m):
    rng = np.random.default_rng(n * 10 + m)
    A = rng.normal(size=(n, n))
    A *= 1.1 / np.abs(np.linalg.eigvals(A)).max()
    B = rng.normal(size=(n, m))
    K, ok = gain.lqr_gain(A, B)
    assert ok
    np.testing.assert_allclose(K, configs.lqr_gain(A, B), rtol=1e-9, atol=1e-11)
    for nn in range(1, 9):
        M = rng.normal(size=(nn, nn))
        assert gain.spectral_radius(M) == pytest.approx(np.abs(np.linalg.eigvals(M)).max(), rel=1e-7)     # (2^30-th root: ~1e-9)


def test_oracle_reports_an_unstabilisable_pair_without_raising():
    """An unstable mode no input reaches: the Riccati doubling diverges, and gain_synthesis reports ok=False with NaN radii."""
    n, m, Tm = 3, 2, 40
    A = np.diag([1.5, 0.5, 0.3])
    B = np.zeros((n, m)); B[1, 0] = 1.0; B[2, 1] = 1.0
    K, ok = gain.lqr_gain(A, B)
    assert not ok
    rng = np.random.default_rng(0)
    Pinv = rng.normal(size=(Tm, n + m)) * 0.01
    r = gain.gain_synthesis(np.hstack([A, B]), Pinv, _wz(n, 3, 1), max_iter=3, num_init=2)
    assert not r["ok"] and np.isnan(r["rho0"]) and np.isnan(r["rho_adv"]) and np.isnan(r["rho_mc"])
    assert not r["robust"]
