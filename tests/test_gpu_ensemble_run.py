"""tz_closed_loop_run_set -- K closed-loop steps of a program set (the data-set axis: one program per data set) in one
launch -- against K calls of tz_closed_loop_step_set on the same inputs: every output of every step bit-equal, for the
three examples (bucket B0) and sets of the larger buckets B1 and B2, cold, warm and with active-set hints, dense and packed
tube, ragged and empty data sets, odd and even batches, with restarts, with a plant per scenario, and for a set with more
tiles than one wave of warps holds.  Also: each data set's slice equals tz_closed_loop_run on that data set's own program,
TZDDPCEnsemble.simulate (which takes the fused run below FUSED_RUN_MAX_BATCH scenarios) equals a written-out step loop,
no write leaves its buffer, and bad arguments are refused."""
import ctypes as C

import numpy as np
import pytest
import torch

import oracle
from tests import common
from tests.test_gpu_guard_bands import Guarded
from tzddpc_b200 import configs

pytestmark = pytest.mark.gpu

TZ_EINVAL = -22          # include/tzddpc.h


def _controllers(cfg, D, horizon=None, seed=0):
    """D controllers of one structure, one per data set (the LQR gain of each data set's model centre)."""
    ctls = []
    for d in range(D):
        u, x = common.dataset(cfg, seed=cfg.seed + 101 * d + seed)
        oo = oracle.OracleTZDDPC(oracle.Data(u, x))
        oo.build_zonotopes(common.oracle_zonotopes(cfg))
        Cm = oo.Mdata.center
        ctls.append(common.make_product(cfg, u, x, configs.lqr_gain(Cm[:, :cfg.n], Cm[:, cfg.n:]), horizon=horizon))
    return ctls


def _inputs(cfg, S, steps, dev, seed):
    """x0 (n, S) and noise (steps, n, S) on the device"""
    rng = np.random.default_rng(seed)
    x0 = np.tile(np.asarray(cfg.X0[0], dtype=np.float64)[:, None], (1, S))
    noise = np.ascontiguousarray(np.transpose(common.noise_for(cfg, steps, S, rng), (0, 2, 1)))
    return torch.tensor(x0, dtype=torch.float64, device=dev), torch.tensor(noise, dtype=torch.float64, device=dev)


def _shared_plant(cfg, dev):
    f64 = dict(dtype=torch.float64, device=dev)
    return (torch.tensor(np.ascontiguousarray(cfg.A, dtype=np.float64), **f64),
            torch.tensor(np.ascontiguousarray(np.asarray(cfg.B, dtype=np.float64).reshape(cfg.n, cfg.m)), **f64))


def _outputs(make, h, steps, S, opts, is_set=True, f64=torch.float64, i32=torch.int32):
    """The per-step outputs of a run of `steps` steps over program set handle h (a program: not is_set), from make(shape, dtype)."""
    from tzddpc_b200 import _abi
    n, m, nv, nt, nent, nnz, warm_rows = _abi.program_dims(h, is_set)
    rows = nnz if opts.tube_packed else nent
    o = dict(status=make((steps, S), i32), iters=make((steps, S), i32), cost=make((steps, S), f64), v=make((steps, nv, S), f64),
             traj=make((steps, nt, S), f64), ze1=make((steps, rows, S), f64), u=make((steps, m, S), f64),
             x_hist=make((steps, n, S), f64), xbar_hist=make((steps, n, S), f64), e_hist=make((steps, n, S), f64),
             stats=make((steps, 8), f64))
    o["warm"] = make((warm_rows, S), f64) if opts.warm_start else None
    return o


def _alloc(dev):
    def make(shape, dtype):
        return torch.zeros(shape, dtype=dtype, device=dev)
    return make


def _loop(h, x0, noise, restart, plant, opts):
    """The reference: one tz_closed_loop_step_set (_plants) launch per step."""
    from tzddpc_b200 import ops
    steps, n, S = noise.shape
    o = _outputs(_alloc(x0.device), h, steps, S, opts)
    x, xb, e = x0.clone(), x0.clone(), torch.zeros_like(x0)
    step = ops.closed_loop_step_set_plants if len(plant) == 1 else ops.closed_loop_step_set
    for k in range(steps):
        step(h, x, xb, e, noise[k], restart, *plant, o["status"][k], o["cost"][k], o["v"][k], o["traj"][k], o["ze1"][k], o["u"][k],
             o["iters"][k], o["warm"], o["stats"][k], opts.pack())
        o["x_hist"][k].copy_(x); o["xbar_hist"][k].copy_(xb); o["e_hist"][k].copy_(e)
    o.update(x=x, xbar=xb, e=e)
    return o


def _run(h, x0, noise, restart, plant, opts, make=None, single=False):
    """tz_closed_loop_run_set (_plants) -- or, with `single`, tz_closed_loop_run on one program -- in one launch."""
    from tzddpc_b200 import ops
    steps, n, S = noise.shape
    make = make or _alloc(x0.device)
    o = _outputs(make, h, steps, S, opts, is_set=not single)
    x, xb, e = make((n, S), torch.float64), make((n, S), torch.float64), make((n, S), torch.float64)
    x.copy_(x0), xb.copy_(x0)
    if single:
        run = ops.closed_loop_run_plants if len(plant) == 1 else ops.closed_loop_run
    else:
        run = ops.closed_loop_run_set_plants if len(plant) == 1 else ops.closed_loop_run_set
    run(h, steps, x, xb, e, noise, restart, *plant, o["status"], o["cost"], o["v"], o["traj"], o["ze1"], o["u"], o["x_hist"],
        o["xbar_hist"], o["e_hist"], o["iters"], o["warm"], o["stats"], opts.pack())
    o.update(x=x, xbar=xb, e=e)
    return o


def _same(a, b, tag, good_only=False):
    """Every output bit for bit (NaN payloads included).  good_only: the values of failed steps (cost, v, traj, tube, u) are
    compared only where the step succeeded -- the rule of tests/test_gpu_fused_run.py, for a step loop that may take the
    two-kernel hot path.  Statistics: to 1e-12 (their sums are accumulated in another order)."""
    torch.cuda.synchronize()
    for k in ("status", "iters", "x_hist", "xbar_hist", "e_hist", "x", "xbar", "e"):
        assert torch.equal(a[k], b[k]), f"{tag}: {k}"
    good = (a["status"] == 0).cpu().numpy()
    for k in ("cost", "v", "traj", "ze1", "u"):
        aa, bb = a[k].cpu().numpy(), b[k].cpu().numpy()
        if good_only:
            g = good if aa.ndim == 2 else np.broadcast_to(good[:, None, :], aa.shape)
            np.testing.assert_array_equal(aa[g], bb[g], err_msg=f"{tag}: {k}")
        else:
            assert np.array_equal(aa.view(np.int64), bb.view(np.int64)), f"{tag}: {k}"
    np.testing.assert_allclose(a["stats"].cpu().numpy(), b["stats"].cpu().numpy(), rtol=1e-12, atol=1e-12, err_msg=f"{tag}: stats")


OPTIONS = [dict(warm_start=0), dict(warm_start=1), dict(warm_start=2), dict(warm_start=2, tube_packed=1),
           dict(warm_start=0, tube_packed=1)]


@pytest.mark.parametrize("name,horizon,counts,steps,bucket", [
    ("double_integrator", None, [16, 16, 16], 12, "B0"),
    ("pulley", None, [32, 0, 16, 7], 9, "B0"),             # an empty data set, a ragged last one, odd S
    ("pulley", None, [16], 5, "B0"),                       # one data set of 16 scenarios
    ("pulley", None, [16, 16], 1, "B0"),                   # one step: one tz_closed_loop_step_set
    ("fivedim", None, [16, 48], 70, "B0"),                 # through the infeasibility wave: restarts
    ("sweep", 3, [16, 32, 9], 6, "B1"),
    ("sweep", 4, [16, 32, 10], 6, "B2"),
])
def test_run_set_equals_the_step_set_loop(cuda_lib, name, horizon, counts, steps, bucket):
    import tzddpc_b200 as tz
    cfg = configs.sweep() if name == "sweep" else configs.CONFIGS[name]()
    ctls = _controllers(cfg, len(counts), horizon=horizon)
    ens = tz.TZDDPCEnsemble(ctls, counts)
    assert ens._program.bucket.startswith(bucket)
    h, S, dev = ens._program.handle.value, ens.num_scenarios, ens.device
    x0, noise = _inputs(cfg, S, steps, dev, seed=len(counts) + steps)
    plant = _shared_plant(cfg, dev)
    restarted = 0
    for kw in OPTIONS:
        opts = tz.SolverOptions(**kw)
        ref = _loop(h, x0, noise, x0, plant, opts)
        got = _run(h, x0, noise, x0, plant, opts)
        _same(ref, got, f"{name} counts={counts} {kw}")
        restarted += int((ref["status"] == 2).sum().item())
        # without x_restart a failed scenario keeps its state
        _same(_loop(h, x0, noise, None, plant, opts), _run(h, x0, noise, None, plant, opts), f"{name} counts={counts} {kw} no restart")
    if name == "fivedim":
        assert restarted > 0, "expected infeasible steps (restarts) in the window"


@pytest.mark.parametrize("warm", [0, 2])
def test_run_set_with_more_tiles_than_a_wave(cuda_lib, warm):
    """120 data sets (cycling through 3 programs) of 256 scenarios: 1,920 tiles, more than one wave of warps (1,776) holds,
    so warps own several rounds of the run.  The step loop at this size takes the hot path with hints (warm 2)."""
    import tzddpc_b200 as tz
    from tzddpc_b200 import _abi
    cfg = configs.CONFIGS["fivedim"]()
    ctls = _controllers(cfg, 3)
    nprog, per, steps = 120, 256, 3
    pset = _abi.ProgramSet([ctls[j % 3]._program for j in range(nprog)], np.arange(nprog + 1, dtype=np.int64) * per)
    S, dev = nprog * per, ctls[0].device
    x0, noise = _inputs(cfg, S, steps, dev, seed=21)
    x0 += 0.01 * torch.randn(x0.shape, generator=torch.Generator(device=dev).manual_seed(3), device=dev, dtype=torch.float64)
    plant = _shared_plant(cfg, dev)
    opts = tz.SolverOptions(warm_start=warm)
    ref = _loop(pset.handle.value, x0, noise, x0, plant, opts)
    got = _run(pset.handle.value, x0, noise, x0, plant, opts)
    _same(ref, got, f"{nprog} x {per} warm {warm}", good_only=warm == 2)
    assert (ref["status"] == 0).float().mean().item() > 0.9


def test_one_step_on_the_hot_path_batch(cuda_lib):
    """nsteps = 1 at a batch where tz_closed_loop_step_set takes the two-kernel hot path: the same step."""
    import tzddpc_b200 as tz
    cfg = configs.CONFIGS["pulley"]()
    ctls = _controllers(cfg, 4)
    ens = tz.TZDDPCEnsemble(ctls, 128)
    h, S, dev = ens._program.handle.value, ens.num_scenarios, ens.device
    x0, noise = _inputs(cfg, S, 3, dev, seed=5)
    plant = _shared_plant(cfg, dev)
    opts = tz.SolverOptions(warm_start=2, hot_path=1)
    ref = _loop(h, x0, noise, x0, plant, opts)          # three steps: the hints of the first make the later ones hot
    x1, xb1, e1 = ref["x_hist"][1].clone(), ref["xbar_hist"][1].clone(), ref["e_hist"][1].clone()
    # step 3 again, alone, from the state and hints the second step left: as a one-step run
    ref2 = _loop(h, x0, noise[:2].contiguous(), x0, plant, opts)
    got = _outputs(_alloc(dev), h, 1, S, opts)
    got["warm"].copy_(ref2["warm"])
    from tzddpc_b200 import ops
    ops.closed_loop_run_set(h, 1, x1, xb1, e1, noise[2:].contiguous(), x0, *plant, got["status"], got["cost"], got["v"], got["traj"],
                            got["ze1"], got["u"], got["x_hist"], got["xbar_hist"], got["e_hist"], got["iters"], got["warm"], got["stats"],
                            opts.pack())
    torch.cuda.synchronize()
    assert torch.equal(got["status"][0], ref["status"][2]) and torch.equal(got["iters"][0], ref["iters"][2])
    for a, b in ((x1, ref["x"]), (xb1, ref["xbar"]), (e1, ref["e"]), (got["x_hist"][0], ref["x_hist"][2])):
        assert torch.equal(a, b)
    good = ref["status"][2] == 0
    assert int(good.sum()) > S // 2
    for k in ("cost", "v", "traj", "ze1", "u"):
        assert torch.equal(got[k][0][..., good], ref[k][2][..., good]), k
    assert int((ref["iters"][2] == 0).sum()) > S // 2, "the hints should decide most scenarios of the third step"


def test_plant_per_scenario(cuda_lib):
    """_run_set_plants with plants drawn from every data set's own model set equals the _step_set_plants loop; with every
    column the shared plant it equals _run_set."""
    import tzddpc_b200 as tz
    cfg = configs.CONFIGS["pulley"]()
    counts = [32, 16, 25]
    ctls = _controllers(cfg, len(counts))
    ens = tz.TZDDPCEnsemble(ctls, counts)
    h, S, dev = ens._program.handle.value, ens.num_scenarios, ens.device
    x0, noise = _inputs(cfg, S, 10, dev, seed=17)
    A, B = ens.sample_plants(seed=9)
    AB = ens._plant_batch(A, B, S)
    assert len(AB) == 1 and not torch.equal(AB[0][:, 0], AB[0][:, 1])
    At, Bt = _shared_plant(cfg, dev)
    AB_shared = ens._plant_batch(At.expand(S, -1, -1), Bt.expand(S, -1, -1), S)
    for kw in (dict(warm_start=2), dict(warm_start=0, tube_packed=1), dict(warm_start=1)):
        opts = tz.SolverOptions(**kw)
        _same(_loop(h, x0, noise, x0, AB, opts), _run(h, x0, noise, x0, AB, opts), f"sampled plants {kw}")
        _same(_run(h, x0, noise, x0, (At, Bt), opts), _run(h, x0, noise, x0, AB_shared, opts), f"shared plant per column {kw}")


@pytest.mark.parametrize("name,counts", [("fivedim", [16, 48, 33]), ("double_integrator", [16, 0, 32])])
def test_each_data_set_equals_its_own_program_run(cuda_lib, name, counts):
    import tzddpc_b200 as tz
    cfg = configs.CONFIGS[name]()
    ctls = _controllers(cfg, len(counts))
    ens = tz.TZDDPCEnsemble(ctls, counts)
    h, S, dev = ens._program.handle.value, ens.num_scenarios, ens.device
    steps = 20
    x0, noise = _inputs(cfg, S, steps, dev, seed=2)
    plant = _shared_plant(cfg, dev)
    for kw in (dict(warm_start=2), dict(warm_start=0, tube_packed=1)):
        opts = tz.SolverOptions(**kw)
        got = _run(h, x0, noise, x0, plant, opts)
        torch.cuda.synchronize()
        for d, c in enumerate(ctls):
            b0, b1 = int(ens.begin[d]), int(ens.begin[d + 1])
            if b1 == b0:
                continue
            sl = slice(b0, b1)
            xd, nd = x0[:, sl].contiguous(), noise[:, :, sl].contiguous()
            rd = _run(c._program.handle.value, xd, nd, xd, plant, opts, single=True)
            one = {k: (v[..., sl].contiguous() if k not in ("stats", "warm") else v) for k, v in got.items() if v is not None}
            rd["stats"] = one["stats"]                  # (the set's statistics sum over every data set)
            _same(rd, one, f"{name} data set {d} {kw}")


@pytest.mark.parametrize("plants", [False, True])
def test_ensemble_simulate_takes_the_fused_run_and_equals_a_step_loop(cuda_lib, plants):
    """TZDDPCEnsemble.simulate below FUSED_RUN_MAX_BATCH scenarios is one tz_closed_loop_run_set launch; its arrays equal a
    step loop of closed_loop_step_set (_plants) written out here, on the same x0, noise and plants."""
    import tzddpc_b200 as tz
    from tzddpc_b200 import ops
    cfg = configs.CONFIGS["pulley"]()
    counts = [48, 16, 21]
    ctls = _controllers(cfg, len(counts))
    ens = tz.TZDDPCEnsemble(ctls, counts)
    S, dev, n, steps = ens.num_scenarios, ens.device, cfg.n, 15
    assert ens._fused_run_ok(S, steps) and not ens._fused_run_ok(S, 1) and not ens._fused_run_ok(256, steps)
    x0n = np.tile(np.asarray(cfg.X0[0], dtype=np.float64), (S, 1))
    noise = common.noise_for(cfg, steps, S, np.random.default_rng(30))         # (steps, S, n)
    A, B = ens.sample_plants(seed=2) if plants else (cfg.A, cfg.B)
    for kw in (dict(warm_start=2), dict(tube_packed=1)):
        opts = tz.SolverOptions(**kw)
        r = ens.simulate(A, B, x0n, noise, keep_tubes=True, restart=True, options=opts)
        # ---- the step loop
        plant = ens._plant_batch(A, B, S)
        x0, w = ens._t(x0n.T), ens._t(np.transpose(noise, (0, 2, 1)))
        ref = _loop(ens._program.handle.value, x0, w, x0, plant, opts)
        torch.cuda.synchronize()
        xs = torch.cat([x0[None], ref["x_hist"]])
        xbs = torch.cat([x0[None], ref["xbar_hist"]])
        es = torch.cat([torch.zeros_like(x0)[None], ref["e_hist"]])
        want = {"x": xs, "xbar": xbs, "e": es, "u": ref["u"], "v": ref["v"]}
        for k, v in want.items():
            assert np.array_equal(r[k], v.permute(0, 2, 1).cpu().numpy()), f"plants={plants} {kw}: {k}"
        for k in ("cost", "status", "iters"):
            assert np.array_equal(r[k], ref[k].cpu().numpy(), equal_nan=k == "cost"), f"plants={plants} {kw}: {k}"
        np.testing.assert_allclose(r["stats"], ref["stats"].cpu().numpy(), rtol=1e-12, atol=1e-12)
        g1 = ens.controllers[0]._program.compiled.g1
        if opts.tube_packed:
            dense = np.zeros((steps, S, n * (1 + g1)))
            dense[:, :, ens._program.tube_pattern] = ref["ze1"].permute(0, 2, 1).cpu().numpy()
            tubes = dense.reshape(steps, S, n, 1 + g1)
        else:
            tubes = ref["ze1"].reshape(steps, n, 1 + g1, S).permute(0, 3, 1, 2).cpu().numpy()
        assert np.array_equal(r["tubes"], tubes, equal_nan=True), f"plants={plants} {kw}: tubes"
        _ = ops


@pytest.mark.parametrize("name,counts,plants", [("fivedim", [16, 0, 37], False), ("pulley", [32, 16], True),
                                                ("double_integrator", [16, 16, 16, 5], False)])
def test_run_set_stays_inside_its_buffers(cuda_lib, name, counts, plants):
    """Every per-step output, history, state and scratch buffer of the run is a window in a sentinel-filled allocation; no
    byte outside the windows changes (dense and packed tube, cold, warm and with hints, restarts)."""
    import tzddpc_b200 as tz
    cfg = configs.CONFIGS[name]()
    ctls = _controllers(cfg, len(counts))
    ens = tz.TZDDPCEnsemble(ctls, counts)
    h, S, dev = ens._program.handle.value, ens.num_scenarios, ens.device
    steps = 40 if name == "fivedim" else 8
    x0, noise = _inputs(cfg, S, steps, dev, seed=13)
    for kw in (dict(warm_start=2), dict(warm_start=2, tube_packed=1), dict(warm_start=1), dict(warm_start=0, tube_packed=1)):
        opts = tz.SolverOptions(**kw)
        g = Guarded(dev)
        make = lambda shape, dtype: g.make(shape, dtype)                  # noqa: E731
        if plants:
            A, B = ens.sample_plants(seed=1)
            plant = (g.make(tuple(ens._plant_batch(A, B, S)[0].shape), init=ens._plant_batch(A, B, S)[0]),)
        else:
            At, Bt = _shared_plant(cfg, dev)
            plant = (g.make(tuple(At.shape), init=At), g.make(tuple(Bt.shape), init=Bt))
        xr = g.make(tuple(x0.shape), init=x0)
        nz = g.make(tuple(noise.shape), init=noise)
        o = _run(h, x0, nz, xr, plant, opts, make=make)
        torch.cuda.synchronize()
        g.check(f"{name} counts={counts} {kw}")
        ref = _loop(h, x0, noise, x0, tuple(p.clone() for p in plant), opts)
        _same(ref, o, f"{name} counts={counts} {kw} (guarded)")


def test_bad_arguments_are_refused(cuda_lib):
    import tzddpc_b200 as tz
    from tzddpc_b200 import _abi, ops
    cfg = configs.CONFIGS["pulley"]()
    ctls = _controllers(cfg, 2)
    ens = tz.TZDDPCEnsemble(ctls, [16, 16])
    h, S, dev = ens._program.handle.value, ens.num_scenarios, ens.device
    x0, noise = _inputs(cfg, S, 2, dev, seed=1)
    opts = tz.SolverOptions()
    o = _outputs(_alloc(dev), h, 2, S, opts)
    x, xb, e = x0.clone(), x0.clone(), torch.zeros_like(x0)
    At, Bt = _shared_plant(cfg, dev)
    p = lambda t: None if t is None else C.c_void_p(t.data_ptr())      # noqa: E731
    L = _abi.lib()
    co = ops._opts(opts.pack())

    def call(fn, S_, nsteps, plant):
        return fn(C.c_void_p(h), C.byref(co), S_, nsteps, p(x), p(xb), p(e), p(noise), None, *map(p, plant), p(o["cost"]), p(o["v"]),
                  None, None, p(o["u"]), None, None, None, p(o["status"]), p(o["iters"]), None, None, None)

    AB = ens._plant_batch(At.expand(S, -1, -1), Bt.expand(S, -1, -1), S)
    for fn, plant in ((L.tz_closed_loop_run_set, (At, Bt)), (L.tz_closed_loop_run_set_plants, AB)):
        assert call(fn, S, 0, plant) == TZ_EINVAL and "nsteps" in _abi.last_error()
        assert call(fn, S, -3, plant) == TZ_EINVAL
        assert call(fn, S - 16, 2, plant) == TZ_EINVAL and "created for" in _abi.last_error()
        assert call(fn, S, 2, plant) == _abi.TZ_OK
    assert L.tz_closed_loop_run_set(None, C.byref(co), S, 2, *([None] * 20)) == TZ_EINVAL
    torch.cuda.synchronize()
    # the ops: a wrong batch reaches the library's check, a wrong AB_true shape is caught before any launch
    with pytest.raises(RuntimeError, match="created for"):
        ops.closed_loop_run_set(h, 2, x[:, :16].contiguous(), xb[:, :16].contiguous(), e[:, :16].contiguous(), noise[:, :, :16].contiguous(),
                                None, At, Bt, o["status"][:, :16].contiguous(), None, None, None, None, None, None, None, None, None,
                                None, None, opts.pack())
    with pytest.raises(AssertionError, match="AB_true"):
        ops.closed_loop_run_set_plants(h, 2, x, xb, e, noise, None, AB[0][:, :S - 1].contiguous(), o["status"], None, None, None, None,
                                       None, None, None, None, None, None, None, opts.pack())
