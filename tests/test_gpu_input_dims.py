"""Every native path at two to four inputs, horizon one and up to four noise generators, against the oracle and exact
references (GPU).

Random systems of tests/test_oracle_input_dims.random_config.  The host canonicaliser builds these programs, and the
step kernels serve them from the buckets observed on a B200 (each test asserts its bucket, so a shape that drifts to
another path fails instead of silently covering something else):

    n, m, N, gW   | nv | nz | nc | bucket
    3, 2, 1, 1    |  2 |  2 |  3 | B0 (fast_step_kernel with two inputs)
    5, 2, 1, 1    |  2 |  2 |  3 | B0
    4, 3, 2, 1    |  6 |  9 | 26 | B3
    6, 3, 2, 3    |  6 |  9 | 30 | B3
    8, 4, 2, 1    |  8 | 12 | 39 | B4: its rows fit B3, its tables (25 KiB) not the 24 KiB B3 stages (largest n, m)
    7, 2, 2, 2    |  4 |  6 | 27 | B2
    4, 4, 3, 1    | 12 | 16 | 49 | B4 (big_step_kernel)
    3, 4, 4, 1    | 16 | 27 | 75 | B4, nv = 16 (the ABI maximum), m > n
    2, 4, 4, 4    | 16 | 26 | 67 | B4, m > n

Only uniquely determined outputs are compared with the oracle (quirk Q7: v_(N-1) enters only the constraints, horizon 1 is a
pure feasibility problem, v_0 is unique only for N >= 2 and m <= n): status, cost, xbar[1] (N >= 2), and Ze[1] evaluated by
the oracle at the kernel's own v.  The kernel's v is a certificate on the oracle's program: feasible to 1e-7 and optimal to
COST_RTOL.  The closed-loop update u = K e + v_0, x+ = A x + B u + w is recomputed exactly on the host.
"""
import numpy as np
import pytest
import torch

from oracle import gain
from tests import common, plants_ref
from tests.test_gpu_guard_bands import Guarded
from tests.test_gpu_plants import _check_guarantee
from tests.test_oracle_input_dims import SHAPES, build, evaluate_program, random_config, sample_points, shape_seed
from tzddpc_b200 import _abi, configs

pytestmark = pytest.mark.gpu

BUCKET = {(3, 2, 1, 1): "B0", (5, 2, 1, 1): "B0", (4, 3, 2, 1): "B3", (6, 3, 2, 3): "B3", (8, 4, 2, 1): "B4", (7, 2, 2, 2): "B2",
          (4, 4, 3, 1): "B4", (3, 4, 4, 1): "B4", (2, 4, 4, 4): "B4", (4, 4, 2, 1): "B3"}
KEYS = ("x", "xbar", "e", "u", "v", "cost", "status", "iters", "tubes")
_CACHE = {}


@pytest.fixture(scope="module")
def ctl(cuda_lib):
    def get(shape):
        if shape not in _CACHE:
            cfg = random_config(*shape, shape_seed(*shape))
            o, K, u, x = build(cfg)
            t = common.make_product(cfg, u, x, K)
            assert t._program.bucket.startswith(BUCKET[shape] + "("), (shape, t._program.bucket)
            _CACHE[shape] = (cfg, o, t)
        return _CACHE[shape]
    return get


def _same(a, b, tag, cols=slice(None)):
    for k in KEYS:
        if k in a:
            np.testing.assert_array_equal(a[k][:, cols], b[k][:, cols], err_msg=f"{tag}: {k}")


def _check_update(out, K, A, B, noise, tag):
    """u_t = K e_t + v_0 and x_(t+1) = A x_t + B u_t + w_t of every feasible step, in float64 on the host, to 1e-14 of the sum
    of the terms' magnitudes.  A (n, n) / B (n, m) shared, or (S, n, n) / (S, n, m) per scenario."""
    m = K.shape[0]
    ok = out["status"] == 0
    assert ok.mean() > 0.5, f"{tag}: too few feasible steps"
    e, x, u, v0 = out["e"][:-1], out["x"], out["u"], out["v"][..., :m]
    ur = np.einsum("ij,tsj->tsi", K, e) + v0
    us = np.einsum("ij,tsj->tsi", np.abs(K), np.abs(e)) + np.abs(v0)
    bad = (np.abs(u - ur) > 1e-14 * us).any(axis=-1) & ok
    assert not bad.any(), f"{tag}: u != K e + v0 at {np.argwhere(bad)[:5]}"
    sub = "ij" if A.ndim == 2 else "sij"
    xr = np.einsum(f"{sub},tsj->tsi", A, x[:-1]) + np.einsum(f"{sub},tsj->tsi", B, u) + noise
    xs = np.einsum(f"{sub},tsj->tsi", np.abs(A), np.abs(x[:-1])) + np.einsum(f"{sub},tsj->tsi", np.abs(B), np.abs(u)) + np.abs(noise)
    bad = (np.abs(x[1:] - xr) > 1e-14 * xs).any(axis=-1) & ok
    assert not bad.any(), f"{tag}: x+ != A x + B u + w at {np.argwhere(bad)[:5]}"


@pytest.mark.parametrize("shape", list(SHAPES))
def test_solve_matches_the_oracle(ctl, shape):
    cfg, o, t = ctl(shape)
    S = 24
    xb, e = sample_points(cfg, S, 3)
    cost, v, xbar, tube, status = t.solve(xb, e)
    Z = tube.Z.value
    wmax = t._program.compiled.wmax
    n_ok = 0
    for i in range(S):
        r = o.solve_status(xb[i], e[i])
        assert (r.status == 2) == (status[i] == 2), (i, r.status, status[i])
        if r.status == 2:
            continue
        n_ok += 1
        assert status[i] == 0
        assert common.cost_close(cost[i], r.cost, wmax), (i, cost[i], r.cost)
        if cfg.horizon >= 2:
            # (at horizon 4 the oracle's interior point stops up to ~4e-7 relative short of the optimal cost, and xbar[1]
            #  moves with the square root of that: tests/test_oracle_input_dims.py)
            tol = 1e-6 if cfg.horizon < 4 else 3e-5
            np.testing.assert_allclose(xbar[i, 1], r.xbar[1], rtol=tol, atol=tol)
        np.testing.assert_allclose(Z[i], o.evaluate_tube(xb[i], e[i], v[i].ravel(), 1), rtol=common.GEN_RTOL, atol=1e-12)
        obj, viol = evaluate_program(o, xb[i], e[i], v[i])
        assert viol <= 1e-7, (i, viol)
        assert common.cost_close(obj, r.cost, wmax), (i, obj, r.cost)
    assert n_ok >= S // 2, f"only {n_ok} feasible points"
    assert n_ok < S, "no infeasible point: the sample does not reach the boundary"


@pytest.mark.parametrize("shape", list(SHAPES))
def test_closed_loop(ctl, shape, monkeypatch):
    import tzddpc_b200 as tz
    for k in ("TZDDPC_FAST_TPB", "TZDDPC_FAST_H", "TZDDPC_FAST_SET_H"):
        monkeypatch.delenv(k, raising=False)
    cfg, o, t = ctl(shape)
    n, m, N = cfg.n, cfg.m, cfg.horizon
    K = t.theta.K
    S, steps = 1000, 8
    rng = np.random.default_rng(shape_seed(*shape))
    noise = common.noise_for(cfg, steps, S, rng)
    x0 = rng.uniform(-0.5, 0.5, size=(S, n))
    pat = t._program.tube_pattern
    runs = {}
    for ws, hot in ((0, 0), (2, 0), (2, 1)):
        for packed in (0, 1):
            out = t.simulate(cfg.A, cfg.B, x0, noise, keep_tubes=True, restart=True,
                             options=tz.SolverOptions(warm_start=ws, hot_path=hot, tube_packed=packed))
            _check_update(out, K, cfg.A, cfg.B, noise, f"{shape} ws={ws} hot={hot} packed={packed}")
            runs[ws, hot, packed] = out
    for packed in (0, 1):                                   # the hot path (B0: fast_step_kernel) against the ADMM kernel
        _same(runs[2, 1, packed], runs[2, 0, packed], f"{shape} hot_path packed={packed}")
    for ws, hot in ((0, 0), (2, 0), (2, 1)):                # packed against dense tube
        d, p = runs[ws, hot, 0], runs[ws, hot, 1]
        for k in KEYS[:-1]:
            np.testing.assert_array_equal(d[k], p[k], err_msg=f"{shape} packed ws={ws} hot={hot}: {k}")
        ok = d["status"] == 0
        flat = lambda a: a.reshape(steps, S, -1)[..., pat][ok]          # noqa: E731
        np.testing.assert_array_equal(flat(d["tubes"]), flat(p["tubes"]))
    # a plant per scenario, from the data-consistent model set
    A3, B3 = (a.cpu().numpy() for a in t.sample_plants(S, seed=5))
    for ws in (0, 2):
        out = t.simulate(A3, B3, x0, noise, keep_tubes=True, restart=True, options=tz.SolverOptions(warm_start=ws))
        _check_update(out, K, A3, B3, noise, f"{shape} plants ws={ws}")
    # small batches: the fused run (buckets <= 3) against the step loop, shared plant and a plant per scenario
    Sf = 7
    if BUCKET[shape] != "B4":
        for A_, B_ in ((cfg.A, cfg.B), (A3[:Sf], B3[:Sf])):
            for opts in (tz.SolverOptions(warm_start=2), tz.SolverOptions(tube_packed=1)):
                assert t._fused_run_ok(Sf, steps)
                fused = t.simulate(A_, B_, x0[:Sf], noise[:, :Sf], keep_tubes=True, restart=True, options=opts)
                t.FUSED_RUN_MAX_BATCH = 0
                try:
                    loop = t.simulate(A_, B_, x0[:Sf], noise[:, :Sf], keep_tubes=True, restart=True, options=opts)
                finally:
                    del t.FUSED_RUN_MAX_BATCH
                _same(fused, loop, f"{shape} fused run")
                _check_update(fused, K, A_, B_, noise[:, :Sf], f"{shape} fused run")
    # the oracle's closed loop, where v_0 is unique
    if m <= n and N >= 2:
        for ws in (0, 2):
            out = t.simulate(cfg.A, cfg.B, x0[:3], noise[:, :3], options=tz.SolverOptions(warm_start=ws))
            for s in range(3):
                rr = o.closed_loop(cfg.A, cfg.B, x0[s], noise[:, s])
                ok = rr["status"] == 0
                last = int(np.argmin(ok)) if not ok.all() else steps
                assert (out["status"][:last, s] == 0).all()
                np.testing.assert_allclose(out["x"][:last + 1, s], rr["x"][:last + 1], rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("shape", [(3, 2, 1, 1), (6, 3, 2, 3), (4, 4, 3, 1)])
def test_the_tube_covers_every_plant_of_msigma(ctl, shape):
    import tzddpc_b200 as tz
    cfg, o, t = ctl(shape)
    S, steps = 4096, 30
    A, B = t.sample_plants(S, seed=31)
    x0 = np.zeros((S, cfg.n))
    kw = dict(steps=steps, seed=32, keep_tubes=True, restart=True, options=tz.SolverOptions(warm_start=2, tube_packed=1))
    out = t.simulate(A, B, x0, **kw)
    _check_guarantee(out, cfg, str(shape))
    # equal plants: bit for bit the shared-plant call
    ref = t.simulate(cfg.A, cfg.B, x0, **kw)
    _same(t.simulate(np.broadcast_to(cfg.A, (S,) + cfg.A.shape).copy(), np.broadcast_to(cfg.B, (S,) + cfg.B.shape).copy(), x0, **kw),
          ref, f"{shape} equal plants")


def test_sampler_and_plant_trajectories_at_four_inputs(cuda_lib):
    from tzddpc_b200 import ops
    cfg = random_config(3, 4, 2, 3, 77)
    u, x = common.dataset(cfg)
    import tzddpc_b200 as tz
    t = tz.TZDDPC(tz.Data(u, x))
    t.verbose = False
    Z = tz.Zonotope
    t.build_zonotopes(tz.SystemZonotopes(Z(*cfg.X0), Z(*cfg.U), Z(*cfg.X), Z(*cfg.W)))
    S, seed, off = 500, 9, 321
    A, B = t.sample_plants(S, seed, off)
    want = plants_ref.sample_plants(t._AB[None], t._Pinv[None].cpu().numpy(), np.asarray(t.zonotopes.W.Z), None, S, seed, off)
    got = torch.cat([A, B], dim=2).cpu().numpy()
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-13 * max(1.0, np.abs(want).max()))
    D, T = 16, 50
    A3, B3 = got[:D, :, :3], got[:D, :, 3:]
    f = lambda a: torch.tensor(np.ascontiguousarray(a, dtype=np.float64), device="cuda")          # noqa: E731
    X0Z = np.hstack([np.full((3, 1), 0.1), 0.2 * np.eye(3)])
    UZ = np.hstack([cfg.U[0][:, None], cfg.U[1]])
    WZ = np.hstack([cfg.W[0][:, None], cfg.W[1]])
    U, X = ops.generate_trajectories(f(A3), f(B3), f(X0Z), f(UZ), f(WZ), D, T, 19, 4)
    Uo, Xo = plants_ref.generate_trajectories_plants(A3, B3, X0Z, UZ, WZ, D, T, 19, 4)
    np.testing.assert_allclose(U.cpu().numpy(), Uo, rtol=0, atol=1e-15)
    np.testing.assert_allclose(X.cpu().numpy(), Xo, rtol=1e-9, atol=1e-12)


def test_dataset_axis_at_three_inputs(cuda_lib):
    """Three data sets of the (6, 3, 2, 3) system in one program set: bit for bit the three controllers' own solves and
    closed-loop steps, with a shared plant and with a plant per scenario."""
    import tzddpc_b200 as tz
    shape = (6, 3, 2, 3)
    cfg = random_config(*shape, shape_seed(*shape))
    ctls = []
    for d in range(3):
        u, x = common.dataset(cfg, seed=cfg.seed + 101 * d)
        o, K = common.make_oracle(cfg, u, x)
        ctls.append(common.make_product(cfg, u, x, K))
        assert ctls[-1]._program.bucket.startswith("B3(")
    per = 48
    ens = tz.TZDDPCEnsemble(ctls, per)
    S = 3 * per
    xb, e = sample_points(cfg, S, 4)
    dev = ens.device
    r = ens.solve_batch(torch.tensor(xb.T.copy(), device=dev), torch.tensor(e.T.copy(), device=dev))
    for d, c in enumerate(ctls):
        sl = slice(d * per, (d + 1) * per)
        rd = c.solve_batch(torch.tensor(xb[sl].T.copy(), device=dev), torch.tensor(e[sl].T.copy(), device=dev))
        for a, b, k in ((rd.status, r.status[sl], "status"), (rd.cost, r.cost[sl], "cost"), (rd.v, r.v[:, sl], "v"),
                        (rd.xbar, r.xbar[:, sl], "xbar"), (rd.tube._ze1, r.tube._ze1[:, sl], "tube")):
            np.testing.assert_array_equal(a.cpu().numpy(), b.cpu().numpy(), err_msg=f"set solve, data set {d}: {k}")   # (NaN: infeasible)
    rng = np.random.default_rng(8)
    x0 = rng.uniform(-0.5, 0.5, size=(S, cfg.n))
    A3, B3 = (a.cpu().numpy() for a in ens.sample_plants(seed=6))
    for ws in (0, 2):
        kw = dict(steps=6, seed=3, keep_tubes=True, restart=True, options=tz.SolverOptions(warm_start=ws))
        shared = ens.simulate(cfg.A, cfg.B, x0, **kw)
        plants = ens.simulate(A3, B3, x0, **kw)
        assert not np.array_equal(shared["x"], plants["x"])
        for d, c in enumerate(ctls):
            sl = slice(d * per, (d + 1) * per)
            _same({k: v[:, sl] for k, v in shared.items() if k in KEYS},
                  c.simulate(cfg.A, cfg.B, x0[sl], scenario_offset=d * per, **kw), f"set, data set {d}, ws={ws}")
            _same({k: v[:, sl] for k, v in plants.items() if k in KEYS},
                  c.simulate(A3[sl], B3[sl], x0[sl], scenario_offset=d * per, **kw), f"set plants, data set {d}, ws={ws}")


# ---------------------------------------------------------------------------------------------------------------- identify
def _identify_data(n, m, gW, Tm, seed):
    rng = np.random.default_rng(seed)
    A = rng.normal(size=(n, n))
    A *= 0.9 / np.abs(np.linalg.eigvals(A)).max()
    B = rng.normal(size=(n, m))
    T = Tm + 1
    U = rng.uniform(-1, 1, size=(2, T, m))
    X = np.zeros((2, T, n))
    X[:, 0] = rng.uniform(-1, 1, size=(2, n))
    for k in range(1, T):
        X[:, k] = X[:, k - 1] @ A.T + U[:, k - 1] @ B.T + 0.05 * rng.uniform(-1, 1, size=(2, n))
    WZ = np.hstack([rng.normal(size=(n, 1)) * 0.01, rng.normal(size=(n, gW)) * 0.02])
    K = rng.normal(size=(2, m, n)) * 0.3
    return X, U, WZ, K


@pytest.mark.parametrize("n,m,gW", [(8, 4, 4), (7, 3, 2), (1, 4, 1), (3, 4, 3)])
def test_identify_at_large_dimensions(cuda_lib, n, m, gW):
    """d = n + m up to 12 (19 of the 20 simultaneous CTA sums), just below and above the dynamic-shared-memory opt-in, the
    longest data set inside 200 KiB and one past it."""
    from tzddpc_b200 import ops
    row = 8 * (3 * n + 2 * m)                               # staged bytes per sample: D', X1c, Y
    below, top = 40960 // row, 200 * 1024 // row
    g = lambda a: torch.tensor(np.ascontiguousarray(a), device="cuda")          # noqa: E731
    for Tm in (below, below + 1, top):
        X, U, WZ, K = _identify_data(n, m, gW, Tm, Tm)
        AB, dAB, dK, Pinv, status = ops.identify(g(X), g(U), g(WZ), g(K), True)
        assert status.cpu().numpy().tolist() == [0, 0]
        gw = np.abs(WZ[:, 1:]).sum(axis=1)
        for s in range(2):
            D = np.vstack([X[s, :-1].T, U[s, :-1].T])
            X1c = X[s, 1:] - WZ[:, 0][None]
            ABref = np.linalg.lstsq(D.T, X1c, rcond=None)[0].T
            Pref = np.linalg.pinv(D)
            np.testing.assert_allclose(AB[s].cpu().numpy(), ABref, rtol=common.GEN_RTOL, atol=common.GEN_RTOL * np.abs(ABref).max())
            P = Pinv[s].cpu().numpy()
            np.testing.assert_allclose(P, Pref, rtol=common.GEN_RTOL, atol=common.GEN_RTOL * np.abs(Pref).max())
            np.testing.assert_allclose(dAB[s].cpu().numpy(), np.outer(gw, np.abs(P).sum(axis=0)), rtol=1e-13)
            np.testing.assert_allclose(dK[s].cpu().numpy(), np.outer(gw, np.abs(P[:, :n] + P[:, n:] @ K[s]).sum(axis=0)), rtol=1e-13)
    X, U, WZ, K = _identify_data(n, m, gW, top + 1, 1)
    with pytest.raises(Exception, match="too long for shared memory"):
        ops.identify(g(X), g(U), g(WZ), g(K), True)


def test_identify_flags_two_equal_inputs(cuda_lib):
    from tzddpc_b200 import ops
    X, U, WZ, K = _identify_data(3, 4, 2, 80, 2)
    U[1, :, 2] = U[1, :, 1]
    g = lambda a: torch.tensor(np.ascontiguousarray(a), device="cuda")          # noqa: E731
    *_, status = ops.identify(g(X), g(U), g(WZ), g(K), False)
    assert status.cpu().numpy().tolist() == [0, _abi.TZ_STATUS_NONFINITE]


# -------------------------------------------------------------------------------------------------------------------- gain
def _gain_models(n, m, gW, Tm, P, seed):
    """P data sets of a random (n, m) system: centres AB (P, n, n+m) and pseudo-inverses (P, Tm, n+m) in numpy."""
    rng = np.random.default_rng(seed)
    A = rng.normal(size=(n, n))
    A *= 1.05 / np.abs(np.linalg.eigvals(A)).max()
    B = rng.normal(size=(n, m))
    ABs, Ps = [], []
    for _ in range(P):
        U = rng.uniform(-1, 1, size=(Tm + 1, m))
        X = np.zeros((Tm + 1, n))
        for k in range(1, Tm + 1):
            X[k] = A @ X[k - 1] + B @ U[k - 1] + 0.05 * rng.uniform(-1, 1, n)
        D = np.vstack([X[:-1].T, U[:-1].T])
        Pinv = np.linalg.pinv(D)
        ABs.append(X[1:].T @ Pinv)
        Ps.append(Pinv)
    GW = rng.normal(size=(n, gW))
    return np.stack(ABs), np.stack(Ps), GW


# (n, m, gW, T-1, the noise scale at which the adversary destabilises the first gain and the outer loop iterates)
GAIN_SHAPES = [(1, 2, 3, 40, 0.6), (3, 3, 4, 40, 0.6), (7, 4, 3, 40, 5.0), (8, 2, 4, 40, 0.6), (3, 4, 3, 600, 5.0)]


@pytest.mark.parametrize("n,m,gW,Tm,big", GAIN_SHAPES)
@pytest.mark.parametrize("inflated", [False, True])
def test_gain_synthesis_and_adversary(cuda_lib, n, m, gW, Tm, big, inflated):
    """64 data sets (8 distinct ones, tiled) with a non-zero dataset_offset: data set d draws from (seed, offset + d).
    The inflated noise zonotope makes the outer loop iterate."""
    from tzddpc_b200 import ops
    scale = big if inflated else 0.02
    ABu, Pu, GW = _gain_models(n, m, gW, Tm, 8, 10 * n + m + Tm)
    WZ = np.hstack([np.zeros((n, 1)), scale * GW / np.abs(GW).max()])
    D, off, seed = 64, 1000, 25
    AB, Pinv = ABu[np.arange(D) % 8], Pu[np.arange(D) % 8]
    if Tm == 600:
        assert Tm * (2 * n + m) * 8 + 4 * gW * Tm + 16 > 40 * 1024          # the opt-in staging branch
    g = lambda a: torch.tensor(np.ascontiguousarray(a), device="cuda")          # noqa: E731
    kw = dict(tol=1e-5, max_iter=6, num_init=4, accuracy=0.03, confidence=1e-2)
    K, dA, dB, rho, robust, iters, status = (a.cpu().numpy() for a in ops.gain_synthesis(
        g(AB), g(Pinv), g(WZ), kw["tol"], kw["max_iter"], kw["num_init"], kw["accuracy"], kw["confidence"], seed, off))
    dA2, dB2, rho2, robust2, status2 = (a.cpu().numpy() for a in ops.gain_adversary(
        g(AB), g(Pinv), g(WZ), g(K), kw["num_init"], kw["accuracy"], kw["confidence"], seed, off))
    iterated = 0
    for d in (0, 1, 9, 37, 63):
        A0, B0 = AB[d][:, :n], AB[d][:, n:]
        r = gain.gain_synthesis(AB[d], Pinv[d], WZ, seed=seed, dataset=off + d, **kw)
        assert bool(status[d] == 0) == r["ok"]
        if not r["ok"]:
            continue
        assert int(iters[d]) == r["iters"]
        iterated += r["iters"] > 0
        np.testing.assert_allclose(K[d], r["K"], rtol=1e-8, atol=1e-10)
        np.testing.assert_allclose(dA[d], r["dA"], rtol=1e-8, atol=1e-11)
        np.testing.assert_allclose(dB[d], r["dB"], rtol=1e-8, atol=1e-11)
        np.testing.assert_allclose(rho[d], [r["rho0"], r["rho_adv"], r["rho_mc"]], rtol=1e-8)
        assert bool(robust[d]) == r["robust"]
        # the radii of the pairs rebuilt from K, dA, dB
        rad = lambda M: np.abs(np.linalg.eigvals(M)).max()          # noqa: E731
        assert rho[d, 0] == pytest.approx(rad(A0 + B0 @ K[d]), rel=1e-7)
        assert rho[d, 1] == pytest.approx(rad(A0 + dA[d] + (B0 + dB[d]) @ K[d]), rel=1e-7)
        if r["iters"] == 0:
            np.testing.assert_allclose(K[d], configs.lqr_gain(A0, B0), rtol=1e-9, atol=1e-9 * np.abs(K[d]).max())
        # tz_gain_adversary with the synthesised gain: one adversary pass and the robustness check
        An, Bn, _ = gain.adversary(A0, B0, Pinv[d], WZ[:, 1:], K[d], kw["num_init"], seed, off + d)
        np.testing.assert_allclose(dA2[d], An - A0, rtol=1e-8, atol=1e-11)
        np.testing.assert_allclose(dB2[d], Bn - B0, rtol=1e-8, atol=1e-11)
        rob, worst, _ = gain.robust_check(A0, B0, Pinv[d], WZ[:, 1:], K[d], kw["accuracy"], kw["confidence"], seed, off + d)
        np.testing.assert_allclose(rho2[d], [gain.spectral_radius(A0 + B0 @ K[d]), gain.spectral_radius(An + Bn @ K[d]), worst], rtol=1e-8)
        assert status2[d] == 0 and bool(robust2[d]) == rob
    # data set d and d + 8 share their model but not their random stream
    assert not np.array_equal(rho[1, 2], rho[9, 2]) or not np.array_equal(rho2[1, 2], rho2[9, 2])
    if inflated:
        assert iterated > 0, "the inflated noise zonotope was meant to exercise the outer loop"


def test_adversary_against_brute_force(cuda_lib):
    """2 gW (T-1) = 12 sign variables: the adversary's objective lies between the centre's and the brute-force maximum."""
    import itertools
    from tzddpc_b200 import ops
    n, m, gW, Tm = 3, 2, 3, 2
    rng = np.random.default_rng(4)
    A0 = rng.normal(size=(n, n)) * 0.5
    B0 = rng.normal(size=(n, m))
    Pinv = rng.normal(size=(Tm, n + m))
    GW = rng.normal(size=(n, gW)) * 0.3
    K = rng.normal(size=(m, n)) * 0.3
    WZ = np.hstack([np.zeros((n, 1)), GW])
    g = lambda a: torch.tensor(np.ascontiguousarray(a), device="cuda")          # noqa: E731
    D = 8
    dA, dB, rho, robust, status = (a.cpu().numpy() for a in ops.gain_adversary(
        g(np.repeat(np.hstack([A0, B0])[None], D, 0)), g(np.repeat(Pinv[None], D, 0)), g(WZ), g(np.repeat(K[None], D, 0)),
        3, 0.1, 0.1, 7, 5))
    assert (status == 0).all()
    PA, PBK = Pinv[:, :n], Pinv[:, n:] @ K
    F0 = A0 + B0 @ K
    best = -np.inf
    for signs in itertools.product((-1.0, 1.0), repeat=2 * gW * Tm):
        s = np.array(signs)
        bA, bB = s[:gW * Tm].reshape(gW, Tm), s[gW * Tm:].reshape(gW, Tm)
        F = F0 - GW @ (bA @ PA + bB @ PBK)
        best = max(best, float((F * F).sum()))
    centre = float((F0 * F0).sum())
    for d in range(D):
        F = A0 + dA[d] + (B0 + dB[d]) @ K
        f = float((F * F).sum())
        assert centre - 1e-12 <= f <= best * (1 + 1e-12), (d, centre, f, best)


def test_unstabilisable_pair_is_reported(cuda_lib):
    from tzddpc_b200 import ops
    n, m, Tm = 3, 2, 40
    A = np.diag([1.5, 0.5, 0.3])
    B = np.zeros((n, m)); B[1, 0] = 1.0; B[2, 1] = 1.0
    rng = np.random.default_rng(0)
    Pinv = rng.normal(size=(Tm, n + m)) * 0.01
    WZ = np.hstack([np.zeros((n, 1)), rng.normal(size=(n, 3)) * 0.02])
    g = lambda a: torch.tensor(np.ascontiguousarray(a), device="cuda")          # noqa: E731
    K, dA, dB, rho, robust, iters, status = ops.gain_synthesis(g(np.hstack([A, B])[None]), g(Pinv[None]), g(WZ), 1e-5, 3, 2, 0.1,
                                                               0.1, 25, 0)
    assert int(status[0]) == _abi.TZ_STATUS_NONFINITE and bool(torch.isnan(rho[0]).all()) and int(robust[0]) == 0
    assert not gain.gain_synthesis(np.hstack([A, B]), Pinv, WZ, max_iter=3, num_init=2)["ok"]


# -------------------------------------------------------------------------------------------------------------- guard bands
@pytest.mark.parametrize("shape,S", [((4, 4, 2, 1), 37), ((8, 4, 2, 1), 9)])
def test_guard_bands_at_four_inputs(ctl, shape, S):
    import tzddpc_b200 as tz
    from tzddpc_b200 import ops
    cfg, o, t = ctl(shape)
    prog = t._program
    n, m, N, g1, nv = cfg.n, cfg.m, cfg.horizon, prog.compiled.g1, prog.compiled.nv
    nent, nt, nnz = n * (1 + g1), (N + 1) * n, len(prog.tube_pattern)
    dev = t.device
    f64 = dict(dtype=torch.float64, device=dev)
    rng = np.random.default_rng(2)
    noise = np.ascontiguousarray(np.transpose(common.noise_for(cfg, 3, S, rng), (0, 2, 1)))
    x0 = rng.uniform(-0.5, 0.5, size=(n, S))
    At = torch.tensor(np.ascontiguousarray(cfg.A), **f64)
    Bt = torch.tensor(np.ascontiguousarray(cfg.B), **f64)
    A3, B3 = t.sample_plants(S, seed=1)
    AB = torch.cat([A3, B3], dim=2).reshape(S, -1).t().contiguous()
    for plants in (False, True):
        for opts in (tz.SolverOptions(warm_start=2), tz.SolverOptions(warm_start=2, tube_packed=1), tz.SolverOptions()):
            g = Guarded(dev)
            rows = nnz if opts.tube_packed else nent
            dx, dxb, de, dxr = g.make((n, S), init=x0), g.make((n, S), init=x0), g.make((n, S)), g.make((n, S), init=x0)
            status, iters = g.make((S,), torch.int32), g.make((S,), torch.int32)
            cost, v, traj, ze, uu = g.make((S,)), g.make((nv, S)), g.make((nt, S)), g.make((rows, S)), g.make((m, S))
            warm = g.make((prog.warm_rows, S)) if opts.warm_start else None
            stats = g.make((8,))
            ABg = g.make((n * (n + m), S), init=AB)
            for k in range(3):
                w = torch.tensor(noise[k], **f64)
                if plants:
                    ops.closed_loop_step_plants(prog.handle.value, dx, dxb, de, w, dxr, ABg, status, cost, v, traj, ze, uu, iters, warm,
                                                stats, opts.pack())
                else:
                    ops.closed_loop_step(prog.handle.value, dx, dxb, de, w, dxr, At, Bt, status, cost, v, traj, ze, uu, iters, warm,
                                         stats, opts.pack())
                torch.cuda.synchronize()
                g.check(f"{shape} plants={plants} warm={opts.warm_start} packed={opts.tube_packed} step {k}")
            assert bool(torch.isfinite(dx).all()) and int((status == 0).sum()) > 0
            # the solve entry point with the same guarded outputs
            cost, v, traj, ze, st, it = ops.solve(prog.handle.value, t._dims[:3] + [rows], dxb, de, warm, True, opts.pack())
            torch.cuda.synchronize()
            g.check(f"{shape} solve")
