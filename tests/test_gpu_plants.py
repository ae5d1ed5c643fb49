"""A plant per scenario (tz_closed_loop_*_plants) and plants drawn from the data-consistent model set M_Sigma
(tz_sample_plants), on the GPU.

* Equal plants: every dispatch path with a plant per scenario, all columns the shared plant, must give the shared-plant
  call's outputs bit for bit.
* Distinct plants: a scenario on plant p must give bit for bit what the shared-plant call with p gives it, and the oracle's
  closed loop on p.
* The sampler against its numpy restatement (tests/plants_ref.py), split batches and the data-set map.
* The guarantee TZDDPC is built on: for every plant of M_Sigma and noise from W, a feasible step's realised error lies in
  Ze[1] and the state in X.
* Data sets from different systems: each data set's closed loop on the plant that produced its data.
* Guard bands around the new entry points' buffers, and rejected shapes / NULL plants."""
import ctypes as C

import numpy as np
import pytest
import torch

import oracle
from oracle.zono import compute_LTI_matrix_zonotope, concatenate_zonotope
from tests import common, plants_ref
from tzddpc_b200 import configs

pytestmark = pytest.mark.gpu

KEYS = ("x", "xbar", "e", "u", "v", "cost", "status", "iters", "tubes")


def _ctl(name, horizon=None, k0=None):
    cfg = configs.CONFIGS[name]() if name != "sweep" else configs.sweep()
    u, x = common.dataset(cfg)
    o, K = common.make_oracle(cfg, u, x, horizon=horizon, k0=k0)
    return cfg, o, common.make_product(cfg, u, x, K, horizon=horizon, k0=k0)


@pytest.fixture(scope="module", params=["double_integrator", "pulley", "fivedim"])
def example(request, cuda_lib):
    return _ctl(request.param)


def _same(a, b, tag, cols=slice(None)):
    for k in KEYS:
        if k in a:
            np.testing.assert_array_equal(a[k][:, cols], b[k][:, cols], err_msg=f"{tag}: {k}")


def _tiled(cfg, S):
    return np.broadcast_to(cfg.A, (S,) + cfg.A.shape).copy(), np.broadcast_to(cfg.B, (S,) + cfg.B.shape).copy()


def _perturbed(cfg, P, seed, rel=0.02):
    rng = np.random.default_rng(seed)
    A = cfg.A[None] * (1 + rel * rng.uniform(-1, 1, (P,) + cfg.A.shape))
    B = cfg.B[None] * (1 + rel * rng.uniform(-1, 1, (P,) + cfg.B.shape))
    return A, B


# (S, steps, options, launch knobs): the hot path at 256 threads and with helper groups (deferred tiles in the first step),
# the ADMM kernel for everything with every warm start, the fused run below 256 scenarios
PATHS = [(4096, 8, dict(warm_start=2, hot_path=1), dict(TZDDPC_FAST_TPB="256")),
         (1000, 8, dict(warm_start=2, hot_path=1), dict(TZDDPC_FAST_TPB="64", TZDDPC_FAST_H="2")),
         (1000, 8, dict(warm_start=2, hot_path=1), dict()),
         (600, 6, dict(warm_start=0, hot_path=0), dict()),
         (600, 6, dict(warm_start=1, hot_path=0), dict()),
         (600, 6, dict(warm_start=2, hot_path=0), dict()),
         (100, 10, dict(warm_start=2), dict()),
         (98, 10, dict(warm_start=0), dict())]


def _knobs(monkeypatch, knobs):
    for k in ("TZDDPC_FAST_TPB", "TZDDPC_FAST_H", "TZDDPC_FAST_SET_H"):
        monkeypatch.delenv(k, raising=False)
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)


@pytest.mark.parametrize("packed", [0, 1])
def test_equal_plants_give_the_shared_plant_bit_for_bit(example, packed, monkeypatch):
    import tzddpc_b200 as tz
    cfg, o, t = example
    for S, steps, opt, knobs in PATHS:
        _knobs(monkeypatch, knobs)
        x0 = np.tile(np.asarray(cfg.X0[0], dtype=np.float64), (S, 1))
        kw = dict(steps=steps, seed=11, vertex_noise=cfg.noise == "vertex", keep_tubes=True, restart=True,
                  options=tz.SolverOptions(tube_packed=packed, **opt))
        ref = t.simulate(cfg.A, cfg.B, x0, **kw)
        A3, B3 = _tiled(cfg, S)
        got = t.simulate(A3, B3, x0, **kw)
        _same(got, ref, f"S={S} {opt} {knobs} packed={packed}")
        At, Bt = torch.tensor(A3, device=t.device), torch.tensor(B3, device=t.device)
        _same(t.simulate(At, Bt, x0, **kw), ref, f"(CUDA tensors) S={S} {opt}")


def test_fivedim_restart_through_the_infeasibility_wave(cuda_lib, monkeypatch):
    """fivedim runs into infeasible steps and restarts from x0 (the reference's run ends there); the full 200 steps."""
    import tzddpc_b200 as tz
    _knobs(monkeypatch, {})
    cfg, o, t = _ctl("fivedim")
    for S in (2048, 200):
        x0 = np.tile(np.asarray(cfg.X0[0], dtype=np.float64), (S, 1))
        kw = dict(steps=cfg.steps, seed=5, restart=True, keep_tubes=False, options=tz.SolverOptions(warm_start=2))
        ref = t.simulate(cfg.A, cfg.B, x0, **kw)
        assert (ref["status"] == 2).any(), "the run must go through infeasible steps"
        _same(t.simulate(*_tiled(cfg, S), x0, **kw), ref, f"fivedim S={S}")


def test_larger_buckets_and_the_generic_path(cuda_lib):
    import tzddpc_b200 as tz
    for horizon, k0 in ((3, None), (5, None), (10, 1)):
        cfg, o, t = _ctl("sweep", horizon, k0)
        assert not t._program.bucket.startswith("B0")
        for S in (64, 300):
            x0 = np.tile(np.asarray(cfg.X0[0], dtype=np.float64), (S, 1))
            for packed in (0, 1):
                kw = dict(steps=4, seed=2, keep_tubes=True, restart=True, options=tz.SolverOptions(tube_packed=packed))
                ref = t.simulate(cfg.A, cfg.B, x0, **kw)
                _same(t.simulate(*_tiled(cfg, S), x0, **kw), ref, f"{t._program.bucket} S={S} packed={packed}")
                A8, B8 = _perturbed(cfg, 4, horizon)
                blk = np.arange(S) * 4 // S
                got = t.simulate(A8[blk], B8[blk], x0, **kw)
                for p in range(4):
                    rp = t.simulate(A8[p], B8[p], x0, **kw)
                    _same(got, rp, f"{t._program.bucket} plant {p}", cols=blk == p)


def _ensemble(name, D, per, seed=0):
    import tzddpc_b200 as tz
    cfg = configs.CONFIGS[name]()
    ctls = []
    for d in range(D):
        u, x = common.dataset(cfg, seed=cfg.seed + 101 * d + seed)
        oo = oracle.OracleTZDDPC(oracle.Data(u, x))
        oo.build_zonotopes(common.oracle_zonotopes(cfg))
        Cm = oo.Mdata.center
        ctls.append(common.make_product(cfg, u, x, configs.lqr_gain(Cm[:, :cfg.n], Cm[:, cfg.n:])))
    return cfg, ctls, tz.TZDDPCEnsemble(ctls, per)


@pytest.mark.parametrize("per", [16, 128])
def test_program_sets(cuda_lib, per, monkeypatch):
    """16-scenario blocks (two program slots per one-warp CTA) and aligned blocks, hot path and ADMM kernel."""
    import tzddpc_b200 as tz
    _knobs(monkeypatch, {})
    cfg, ctls, ens = _ensemble("pulley", 16 if per == 16 else 4, per)
    S = ens.num_scenarios
    x0 = np.tile(np.asarray(cfg.X0[0], dtype=np.float64), (S, 1))
    A8, B8 = _perturbed(cfg, 8, per)
    blk = np.arange(S) * 8 // S
    for opt in (dict(warm_start=2, hot_path=1), dict(warm_start=2, hot_path=0), dict(warm_start=0)):
        for packed in (0, 1):
            kw = dict(steps=6, seed=8, keep_tubes=True, restart=True, options=tz.SolverOptions(tube_packed=packed, **opt))
            ref = ens.simulate(cfg.A, cfg.B, x0, **kw)
            _same(ens.simulate(*_tiled(cfg, S), x0, **kw), ref, f"set per={per} {opt} packed={packed}")
            got = ens.simulate(A8[blk], B8[blk], x0, **kw)
            for p in range(8):
                _same(got, ens.simulate(A8[p], B8[p], x0, **kw), f"set per={per} {opt} plant {p}", cols=blk == p)


@pytest.mark.parametrize("S,opt", [(2048, dict(warm_start=2, hot_path=1)), (512, dict(warm_start=0)),
                                   (120, dict(warm_start=2))])
def test_distinct_plants_equal_the_shared_call_with_their_plant(example, S, opt, monkeypatch):
    import tzddpc_b200 as tz
    _knobs(monkeypatch, {})
    cfg, o, t = example
    steps = 10
    A8, B8 = _perturbed(cfg, 8, S)
    blk = np.arange(S) * 8 // S
    rng = np.random.default_rng(S)
    noise = common.noise_for(cfg, steps, S, rng)
    x0 = np.tile(np.asarray(cfg.X0[0], dtype=np.float64), (S, 1))
    kw = dict(keep_tubes=True, restart=False, options=tz.SolverOptions(**opt))
    got = t.simulate(A8[blk], B8[blk], x0, noise, **kw)
    assert not np.array_equal(got["x"][:, blk == 0][:, 0], got["x"][:, blk == 1][:, 0])
    for p in range(8):
        _same(got, t.simulate(A8[p], B8[p], x0, noise, **kw), f"S={S} {opt} plant {p}", cols=blk == p)
    wmax = t._program.compiled.wmax
    for s in range(0, S, S // 5):
        r = o.closed_loop(A8[blk[s]], B8[blk[s]], x0[s], noise[:, s], keep_tubes=True)
        assert np.array_equal(got["status"][:, s] == 2, r["status"] == 2)
        ok = r["status"] == 0
        last = int(np.argmin(ok)) if not ok.all() else steps
        np.testing.assert_allclose(got["x"][:last + 1, s], r["x"][:last + 1], rtol=1e-6, atol=1e-6)
        np.testing.assert_allclose(got["u"][:last, s], r["u"][:last], rtol=1e-6, atol=1e-6)
        assert common.cost_close(got["cost"][:last, s], r["cost"][:last], wmax).all()


def test_sampler_matches_numpy_and_does_not_depend_on_the_split(example):
    import tzddpc_b200 as tz
    cfg, o, t = example
    S, seed, off = 3000, 77, 12345
    A, B = t.sample_plants(S, seed, off)
    assert A.shape == (S, cfg.n, cfg.n) and B.shape == (S, cfg.n, cfg.m) and A.is_cuda
    want = plants_ref.sample_plants(t._AB[None], t._Pinv[None].cpu().numpy(), np.asarray(t.zonotopes.W.Z), None, S, seed, off)
    got = torch.cat([A, B], dim=2).cpu().numpy()
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-13 * max(1.0, np.abs(want).max()))
    A1, B1 = t.sample_plants(1000, seed, off)
    A2, B2 = t.sample_plants(S - 1000, seed, off + 1000)
    assert torch.equal(torch.cat([A1, A2]), A) and torch.equal(torch.cat([B1, B2]), B)
    # every sample is a point of M_Sigma (the un-reduced set; its generator box around the centre)
    assert not torch.equal(A[0], A[1])
    Mw = concatenate_zonotope(oracle.Zonotope(*cfg.W), t.num_samples - 1)
    d = t.dataset
    M = compute_LTI_matrix_zonotope(d.Xm, d.Xp, d.Um, Mw)
    for s in range(3):
        assert M.contains(got[s], tol=1e-9)
    _ = tz


def test_sampler_honours_the_dataset_map(cuda_lib):
    import tzddpc_b200 as tz
    from tzddpc_b200 import ops
    cfg, ctls, ens = _ensemble("pulley", 3, 32)
    A, B = ens.sample_plants(seed=4)
    got = torch.cat([A, B], dim=2).cpu().numpy()
    for d, c in enumerate(ctls):
        Ad, Bd = c.sample_plants(32, 4, 32 * d)
        np.testing.assert_array_equal(got[32 * d:32 * (d + 1)], torch.cat([Ad, Bd], dim=2).cpu().numpy())
    ABd = torch.stack([torch.tensor(c._AB, device=ens.device) for c in ctls])
    P = torch.stack([c._Pinv for c in ctls]).contiguous()
    WZ = torch.tensor(np.asarray(ens.zonotopes.W.Z), device=ens.device)
    ds = torch.tensor([2, 0, 1, 1, 0, 2, 7, -1], dtype=torch.int32, device=ens.device)
    out = ops.sample_plants(ABd, P, WZ, ds, 8, 9, 0).t().cpu().numpy()
    want = plants_ref.sample_plants(ABd.cpu().numpy(), P.cpu().numpy(), WZ.cpu().numpy(), np.clip(ds.cpu().numpy(), 0, 2), 8, 9, 0)
    np.testing.assert_allclose(out[:6].reshape(6, cfg.n, -1), want[:6], rtol=0, atol=1e-12)
    assert np.isnan(out[6:]).all()                     # a data set outside [0, D): NaN plant
    _ = tz


def _check_guarantee(out, cfg, tag):
    Xi = oracle.Zonotope(*cfg.X).interval
    st = out["status"]
    Z = out["tubes"]                                   # (steps, S, n, 1+g1): Ze[1] of every step
    e1, x1 = out["e"][1:], out["x"][1:]
    feas = st == 0
    assert feas.mean() > 0.5, f"{tag}: too few feasible steps to say anything"
    c, rad = Z[..., 0], np.abs(Z[..., 1:]).sum(axis=-1)
    viol = (np.abs(e1 - c) > rad + 1e-9).any(axis=-1) & feas
    assert not viol.any(), f"{tag}: e_(t+1) outside Ze[1] at {np.argwhere(viol)[:5]}"
    out_x = ((x1 < Xi.left_limit - 1e-9) | (x1 > Xi.right_limit + 1e-9)).any(axis=-1) & feas
    assert not out_x.any(), f"{tag}: x_(t+1) outside X at {np.argwhere(out_x)[:5]}"


@pytest.mark.parametrize("name", ["double_integrator", "pulley", "fivedim"])
def test_the_tube_covers_every_plant_of_msigma(cuda_lib, name):
    import tzddpc_b200 as tz
    cfg, o, t = _ctl(name)
    S, steps = 4096, 30
    A, B = t.sample_plants(S, seed=31)
    x0 = np.tile(np.asarray(cfg.X0[0], dtype=np.float64), (S, 1))
    out = t.simulate(A, B, x0, steps=steps, seed=32, vertex_noise=cfg.noise == "vertex", keep_tubes=True, restart=True,
                     options=tz.SolverOptions(warm_start=2, tube_packed=1))
    _check_guarantee(out, cfg, name)


def test_the_tube_covers_every_plant_of_each_data_sets_msigma(cuda_lib):
    import tzddpc_b200 as tz
    cfg = configs.CONFIGS["pulley"]()
    D, per = 64, 64
    Z = tz.Zonotope
    zon = tz.SystemZonotopes(Z(*cfg.X0), Z(*cfg.U), Z(*cfg.X), Z(*cfg.W))
    data = [tz.Data(*common.dataset(cfg, seed=cfg.seed + 7 * d)) for d in range(D)]
    K = configs.lqr_gain(cfg.A, cfg.B)
    ens = tz.TZDDPCEnsemble.from_datasets(data, zon, cfg.horizon, tz.StageCost(**cfg.cost), tz.BoxConstraint(),
                                          scenarios_per_dataset=per, K=K)
    A, B = ens.sample_plants(seed=41)
    x0 = np.tile(np.asarray(cfg.X0[0], dtype=np.float64), (D * per, 1))
    out = ens.simulate(A, B, x0, steps=30, seed=42, keep_tubes=True, restart=True, options=tz.SolverOptions(warm_start=2))
    _check_guarantee(out, cfg, "ensemble")


def test_datasets_from_different_systems(cuda_lib):
    import tzddpc_b200 as tz
    from tzddpc_b200 import ops
    cfg = configs.CONFIGS["pulley"]()
    D, per, steps = 64, 16, 12
    A3, B3 = _perturbed(cfg, D, 5)
    dev = torch.device("cuda")
    f = lambda a: torch.tensor(np.ascontiguousarray(a, dtype=np.float64), device=dev)       # noqa: E731
    X0Z = np.hstack([cfg.X0[0][:, None], cfg.X0[1]])
    UZ = np.hstack([cfg.U[0][:, None], cfg.U[1]])
    WZ = np.hstack([cfg.W[0][:, None], cfg.W[1]])
    U, X = ops.generate_trajectories(f(A3), f(B3), f(X0Z), f(UZ), f(WZ), D, cfg.T, 19, 0)
    for d in (0, 17, 63):
        Ud, Xd = ops.generate_trajectories(f(A3[d]), f(B3[d]), f(X0Z), f(UZ), f(WZ), 1, cfg.T, 19, d)
        assert torch.equal(Ud[0], U[d]) and torch.equal(Xd[0], X[d])
    Uo, Xo = plants_ref.generate_trajectories_plants(A3, B3, X0Z, UZ, WZ, D, cfg.T, 19)
    np.testing.assert_allclose(X.cpu().numpy(), Xo, rtol=1e-9, atol=1e-12)
    Z = tz.Zonotope
    zon = tz.SystemZonotopes(Z(*cfg.X0), Z(*cfg.U), Z(*cfg.X), Z(*cfg.W))
    ens = tz.TZDDPCEnsemble.from_datasets((U, X), zon, cfg.horizon, tz.StageCost(**cfg.cost), tz.BoxConstraint(), scenarios_per_dataset=per,
                                          K=configs.lqr_gain(cfg.A, cfg.B))
    ds = ens.dataset_of()
    x0 = np.tile(np.asarray(cfg.X0[0], dtype=np.float64), (D * per, 1))
    for opt in (dict(warm_start=2), dict(warm_start=0)):
        kw = dict(steps=steps, seed=3, restart=True, keep_tubes=True, options=tz.SolverOptions(**opt))
        r = ens.simulate(A3[ds], B3[ds], x0, **kw)
        for d in (0, 1, 30, 63):
            sl = slice(d * per, (d + 1) * per)
            rd = ens.controllers[d].simulate(A3[d], B3[d], x0[sl], scenario_offset=d * per, **kw)
            for k in KEYS:
                np.testing.assert_array_equal(r[k][:, sl], rd[k], err_msg=f"{k}, data set {d}, {opt}")


def test_guard_bands_and_validation(example):
    import tzddpc_b200 as tz
    from tzddpc_b200 import _abi, ops
    cfg, o, t = example
    n, m, S, pad = cfg.n, cfg.m, 1000, 64
    dev = t.device
    sentinel = -1234.5

    def banded(rows, dtype=torch.float64, fill=0.0):
        buf = torch.full((pad + rows * S + pad,), sentinel if dtype == torch.float64 else -77, dtype=dtype, device=dev)
        v = buf[pad:pad + rows * S].view(rows, S)
        v.fill_(fill)
        return buf, v

    def intact(buf, rows):
        return bool((buf[:pad] == buf[0]).all() and (buf[pad + rows * S:] == buf[0]).all())

    A, B = t.sample_plants(S, seed=1)
    AB = torch.cat([A, B], dim=2).reshape(S, -1).t().contiguous()
    abuf, ABv = banded(n * (n + m))
    ABv.copy_(AB)
    x0 = torch.tensor(np.asarray(cfg.X0[0], dtype=np.float64), device=dev)[:, None].expand(n, S).contiguous()
    bufs = {k: banded(r) for k, r in (("x", n), ("xbar", n), ("e", n), ("cost", 1), ("u", m), ("v", t._dims[1]),
                                      ("ze1", t._dims[3]), ("warm", t._program.warm_rows))}
    sbuf, stv = banded(1, torch.int32)
    bufs["x"][1].copy_(x0), bufs["xbar"][1].copy_(x0)
    noise = ops.sample_noise(t._t(t.zonotopes.W.Z), S, False, 3, 0, 0)
    opts = tz.SolverOptions(warm_start=2).pack()
    for _ in range(3):
        ops.closed_loop_step_plants(t._program.handle.value, bufs["x"][1], bufs["xbar"][1], bufs["e"][1], noise, None, ABv, stv[0],
                                    bufs["cost"][1][0], bufs["v"][1], None, bufs["ze1"][1], bufs["u"][1], None, bufs["warm"][1], None,
                                    opts)
    torch.cuda.synchronize()
    for k, (buf, v) in bufs.items():
        assert intact(buf, v.shape[0]), k
    assert intact(sbuf, 1) and intact(abuf, n * (n + m)) and torch.equal(ABv, AB)
    # the sampler's output
    obuf, ov = banded(n * (n + m))
    WZ = t._t(t.zonotopes.W.Z)
    ov.copy_(ops.sample_plants(t._t(t._AB)[None], t._Pinv[None].contiguous(), WZ, None, S, 1, 0))
    L = _abi.lib()
    ABc = t._t(t._AB)
    torch.cuda.synchronize()
    rc = L.tz_sample_plants(S, 1, t._Pinv.shape[0] + 1, n, m, WZ.shape[1] - 1, ABc.data_ptr(), t._Pinv.data_ptr(),
                            WZ.data_ptr(), None, 1, 0, ov.data_ptr(), None)
    torch.cuda.synchronize()
    assert rc == 0 and intact(obuf, n * (n + m)) and torch.equal(ov, AB)
    # wrong shapes and NULL plants are rejected before any launch
    with pytest.raises(AssertionError, match="AB_true"):
        ops.closed_loop_step_plants(t._program.handle.value, bufs["x"][1], bufs["xbar"][1], bufs["e"][1], noise, None, ABv[:-1].contiguous(),
                                    stv[0], None, None, None, None, None, None, None, None, opts)
    with pytest.raises(AssertionError, match="A_true, B_true"):
        t.simulate(A[:-1], B[:-1], np.tile(cfg.X0[0], (S, 1)), steps=2, seed=1)
    with pytest.raises(AssertionError, match="A_true, B_true"):
        t.simulate(A, B[:, :, :0], np.tile(cfg.X0[0], (S, 1)), steps=2, seed=1)
    o_ = _abi.TzSolverOpts()
    L.tz_solver_opts_default(C.byref(o_))
    p = lambda v: C.c_void_p(v.data_ptr())                                                         # noqa: E731
    rc = L.tz_closed_loop_step_plants(t._program.handle, C.byref(o_), S, p(bufs["x"][1]), p(bufs["xbar"][1]), p(bufs["e"][1]), p(noise),
                                      None, None, None, None, None, None, None, p(stv), None, None, None, None)
    assert rc == -22 and "AB_true" in _abi.last_error()
    rc = L.tz_closed_loop_run_plants(t._program.handle, C.byref(o_), S, 2, p(bufs["x"][1]), p(bufs["xbar"][1]), p(bufs["e"][1]), p(noise),
                                     None, None, None, None, None, None, None, None, None, None, p(stv), None, None, None, None)
    assert rc == -22
    rc = L.tz_sample_plants(S, 1, 70000, n, m, 2, p(ov), p(ov), p(WZ), None, 1, 0, p(ov), None)
    assert rc == -22
    rc = L.tz_sample_plants(S, 1, t._Pinv.shape[0] + 1, n, m, WZ.shape[1] - 1, None, None, None, None, 1, 0, None, None)
    assert rc == -22
    rc = L.tz_generate_trajectories_plants(4, 10, n, m, 0, 0, 0, None, None, None, None, None, 1, 0, None, None, None)
    assert rc == -22
    # an ensemble whose controllers carry no pseudo-inverse cannot sample
    c2 = _ctl(cfg.name)[2]
    c2._Pinv = None
    with pytest.raises(RuntimeError, match="pseudo-inverse"):
        tz.TZDDPCEnsemble([c2], 16).sample_plants(seed=1)
    with pytest.raises(RuntimeError, match="pseudo-inverse"):
        c2.sample_plants(4, 1)
