#!/usr/bin/env python
"""Benchmark of the TZDDPC hot path: closed-loop steps/sec over batched scenarios.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload fivedim|pulley|double_integrator]
                    [--scaling strong|weak] [--scenarios S] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A "step" is ONE fused closed-loop step (solve + tube + plant/nominal/error update,
examples/3.5dimsystem_sim.py:73-89) over the whole scenario batch.  Default workload: BASELINE.json configs[3], the 5-dim
system with 65,536 scenarios (noise realisations) SHARDED over the N GPUs ("strong" scaling: contiguous shards, Philox
noise keyed by the global scenario index so that a scenario sees the same realisation however the batch is sharded, no
collective in the loop, one NCCL all-reduce of the closed-loop statistics after it).  `--scaling weak` gives every rank
its own `--scenarios`; at N > 1 the strong run reports the weak number beside it (`weak_scaling`).

Prints ONE JSON line (rank 0).  `value` = scenario-steps/s with all state resident in HBM (dense Ze[1].Z, what the
reference returns); `roofline` = algorithmic HBM bytes (SURVEY.md 8d) over the CUDA-event duration of one step's kernels;
`roofline_packed` = the same with the packed tube (the mode the e2e leg and any caller that does not need the structural
zeros uses); `e2e` = the same metric through the host-buffer C-ABI call (pinned host arrays in, the step's results back on
the host every step); `cpu_baseline` = the CPU oracle port timed here on the same window of the workload.
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "closed-loop TZDDPC steps/sec over batched scenarios"
UNIT = "scenario-steps/s"


def algorithmic_bytes_per_scenario_step(n, m, N, g1, tube_rows=None):
    """SURVEY.md 8(d): read x, xbar, e; write x+, xbar+, e+, v, xbar trajectory, cost, Ze[1].Z, status.
    tube_rows: entries of Ze[1].Z written (default: the dense n(1+g1); the packed tube writes n_nz)."""
    rows = n * (1 + g1) if tube_rows is None else tube_rows
    return 8 * (6 * n + N * m + (N + 1) * n + 1 + rows) + 4


def ncu_evidence(kernel: str):
    """Numbers of the committed `ncu --set full` capture of the dominant kernel (profiles/step_kernel_traffic.json, written
    by profiles/fastsum.py --json): dram bytes per launch, FP64-pipe and issue-slot utilisation.  None when absent."""
    p = os.path.join(ROOT, "profiles", "step_kernel_traffic.json")
    try:
        return json.load(open(p)).get(kernel)
    except Exception:
        return None


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------
# CPU side: the oracle port (the reference itself cannot be imported: cvxpy/pyzonotope are absent)
# ----------------------------------------------------------------------------------------------
def _oracle_setup(workload):
    import oracle
    from tzddpc_b200 import configs
    cfg = configs.CONFIGS[workload]()
    rng = np.random.default_rng(cfg.seed)
    u, x = configs.generate_dataset(cfg, rng)
    Z = oracle.Zonotope
    zon = oracle.SystemZonotopes(Z(*cfg.X0), Z(*cfg.U), Z(*cfg.X), Z(*cfg.W))
    o = oracle.OracleTZDDPC(oracle.Data(u, x))
    o.build_zonotopes(zon)
    C = o.Mdata.center
    K = configs.lqr_gain(C[:, :cfg.n], C[:, cfg.n:])
    o.build_zonotopes_theta(zon, K)
    box = oracle.BoxConstraint(**cfg.box) if cfg.box else None
    o.build_problem(cfg.horizon, oracle.StageCost(**cfg.cost), box)
    return cfg, o


def _oracle_worker(args):
    """Closed loop of `scen` scenarios for warmup+steps steps -- the loop of examples/3.5dimsystem_sim.py:73-89 with the
    reference's `solve` (feasibility verdict included: an infeasible or failed step ends the run, tzddpc/tzddpc.py:366-375,
    and the scenario starts a new run from x0, exactly what the GPU leg does).  Returns seconds spent in the timed steps."""
    workload, scen, warmup, steps, seed = args
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    cfg, o = _oracle_setup(workload)
    rng = np.random.default_rng(seed)
    cW, GW = cfg.W
    K = o.theta.K
    x0 = np.asarray(cfg.X0[0], dtype=np.float64)
    x = np.tile(x0, (scen, 1))
    xbar, e = x.copy(), np.zeros_like(x)
    t_timed = 0.0
    for t in range(warmup + steps):
        w = cW[None] + rng.uniform(-1, 1, size=(scen, GW.shape[1])) @ GW.T
        t0 = time.perf_counter()
        for s in range(scen):
            r = o.solve_status(xbar[s], e[s])
            if r.status != 0:
                x[s], xbar[s], e[s] = x0, x0, 0.0
                continue
            u = K @ e[s] + r.v[0]
            x[s] = cfg.A @ x[s] + cfg.B @ u + w[s]
            xbar[s] = r.xbar[1]
            e[s] = x[s] - xbar[s]
        if t >= warmup:
            t_timed += time.perf_counter() - t0
    return t_timed


def cpu_oracle_throughput(workload, cores, scen_per_core, warmup, steps):
    """scenario-steps/s of the oracle port on `cores` host processes (one per core)."""
    jobs = [(workload, scen_per_core, warmup, steps, 1000 + i) for i in range(cores)]
    if cores == 1:
        times = [_oracle_worker(jobs[0])]
    else:
        import multiprocessing as mp
        with mp.get_context("spawn").Pool(cores) as pool:
            times = pool.map(_oracle_worker, jobs)
    return cores * scen_per_core * steps / max(times), max(times)


def workload_name(cfg, S_total, world, scaling):
    how = (f"{S_total} scenarios sharded over {world} GPU(s)" if scaling == "strong" else f"{S_total // world} scenarios per GPU")
    return f"{cfg.name}: n={cfg.n} m={cfg.m} T={cfg.T} horizon={cfg.horizon}, {how} (noise realisations, shared data set), closed loop"


def total_scenarios(args, world):
    return args.scenarios if args.scaling == "strong" else args.scenarios * world


def run_reference(args):
    """The reference arm: the CPU oracle port on all host cores, on the arm's config / metric / window (steps W .. W+K of the
    closed loop), each step a bounded sample of `--cpu-scen` scenarios per core.  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from tzddpc_b200 import configs
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    cfg = configs.CONFIGS[args.workload]()
    cores = len(os.sched_getaffinity(0))
    scen_per_core = max(1, args.cpu_scen // 8)
    val, secs = cpu_oracle_throughput(args.workload, cores, scen_per_core, args.warmup, args.steps)
    sample = (f"{cores * scen_per_core} scenarios ({scen_per_core} per core) x steps {args.warmup}..{args.warmup + args.steps} of the "
              f"closed loop, one process per core ({secs:.1f} s)")
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(cfg, total_scenarios(args, world), world, args.scaling),
                       "parallelism": f"scenario-dp{world}",
                       "note": "CPU oracle port of the reference path (the reference itself needs cvxpy / pyzonotope / "
                               "pydatadrivenreachability, absent here); each step is a bounded sample of the workload: " + sample},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "per_core": val / cores},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md): NVML polled from a thread every ~2 ms
    (the timed region of the default run lasts tens of milliseconds, too short for `nvidia-smi -lms`)."""

    def __init__(self, device_index):
        self.rows, self.ok, self._stop = [], False, False
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = device_index
            if vis:
                ent = vis.split(",")[device_index].strip()
                if ent.startswith("GPU-"):
                    self.h = pynvml.nvmlDeviceGetHandleByUUID(ent)
                    idx = None
                else:
                    idx = int(ent)
            if idx is not None:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
        except Exception as e:      # noqa: BLE001
            self.err = repr(e)

    def sample(self):
        if not self.ok:
            return
        nv = self.nv
        try:
            self.rows.append((time.perf_counter(), nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM),
                              nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)))
        except Exception:       # noqa: BLE001
            pass

    def _poll(self):
        while not self._stop:
            self.sample()
            time.sleep(0.002)

    def stop(self, t0, t1):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "err", "?")]}
        self._stop = True
        self.th.join(timeout=1.0)
        nv = self.nv
        rows = [r for r in self.rows if t0 <= r[0] <= t1] or self.rows[-3:]
        names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        reasons = sorted(k for k, bit in names.items() if any(r[2] & bit for r in rows))
        sm = [r[1] for r in rows]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(self.max_sm), "reasons": reasons,
                "samples": len(sm)}


def build_controller(tz, configs, cfg, dev, horizon=None, k0=None):
    """Set-up of one controller (not timed in the step legs): identify on the GPU, LQR gain, canonicalise, upload."""
    rng = np.random.default_rng(cfg.seed)
    u_data, x_data = configs.generate_dataset(cfg, rng)
    ctl = tz.TZDDPC(tz.Data(u_data, x_data), device=dev)
    ctl.verbose = False
    Z = tz.Zonotope
    zon = tz.SystemZonotopes(Z(*cfg.X0), Z(*cfg.U), Z(*cfg.X), Z(*cfg.W))
    ctl.build_zonotopes(zon)
    n = cfg.n
    Kgain = configs.lqr_gain(ctl.Mdata.center[:, :n], ctl.Mdata.center[:, n:])
    ctl.build_zonotopes_theta(zon, K=Kgain)
    cost, box = tz.StageCost(**cfg.cost), (tz.BoxConstraint(**cfg.box) if cfg.box else tz.BoxConstraint())
    if k0 is None:
        ctl.build_problem(horizon or cfg.horizon, cost, box)
    else:
        ctl.build_problem_simplified(k0, horizon or cfg.horizon, cost, box)
    return ctl


class ClosedLoop:
    """S scenarios of one controller on one device: state, ring buffers of the per-step outputs, Philox noise keyed by the
    GLOBAL scenario index (shard-invariant), and a `step(t)` that launches one fused closed-loop step."""

    def __init__(self, tz, ops, torch, ctl, cfg, dev, S, offset, nring, opts, seed=25, ablate=0):
        from tzddpc_b200 import _abi
        self.torch, self.ops, self.S, self.cfg, self.dev = torch, ops, S, cfg, dev
        prog = ctl._program
        n, N = cfg.n, cfg.horizon
        self.prog, self.n = prog, n
        g1, nv = prog.compiled.g1, prog.compiled.nv
        self.rows = len(prog.tube_pattern) if opts.tube_packed else n * (1 + g1)
        f64 = dict(dtype=torch.float64, device=dev)
        WZ = torch.tensor(np.hstack([cfg.W[0][:, None], cfg.W[1]]), **f64)
        # w_t = W.sample() (examples/2.pulley_sim.py:92) / a random vertex of W (examples/1.double_integrator_sim.py:85) from the
        # Philox stream (seed, offset + scenario, t): pre-drawn for `nring` steps and cycled (bounded memory for long runs)
        self.noise = torch.stack([ops.sample_noise(WZ, S, cfg.noise == "vertex", seed, offset, t) for t in range(nring)])
        self.nring = nring
        self.x0 = torch.tensor(cfg.X0[0], **f64)[:, None].repeat(1, S).contiguous()
        self.x, self.xbar, self.e = self.x0.clone(), self.x0.clone(), torch.zeros((n, S), **f64)
        self.At, self.Bt = torch.tensor(cfg.A, **f64), torch.tensor(cfg.B, **f64)
        ring = 4
        self.ring = ring
        self.ze1 = torch.empty((ring, self.rows, S), **f64)
        self.traj = torch.empty((ring, (N + 1) * n, S), **f64)
        self.v = torch.empty((ring, nv, S), **f64)
        self.cost = torch.empty((ring, S), **f64)
        self.status = torch.zeros((ring, S), dtype=torch.int32, device=dev)
        self.iters = torch.zeros((ring, S), dtype=torch.int32, device=dev)
        self.warm = torch.zeros((prog.warm_rows, S), **f64) if opts.warm_start else None
        self.stats = None
        self.po, self.h, self.ablate = opts.pack(), prog.handle.value, ablate
        self.nstats = _abi.TZ_NSTATS

    def reset(self, total_steps):
        t = self.torch
        self.x.copy_(self.x0); self.xbar.copy_(self.x0); self.e.zero_()
        if self.warm is not None:
            self.warm.zero_()
        self.stats = t.zeros((total_steps, self.nstats), dtype=t.float64, device=self.dev)

    def step(self, t):
        r = t % self.ring
        self.ops.closed_loop_step(self.h, self.x, self.xbar, self.e, self.noise[t % self.nring], self.x0, self.At, self.Bt,
                                  self.status[r], self.cost[r], self.v[r], None if self.ablate >= 2 else self.traj[r],
                                  None if self.ablate >= 1 else self.ze1[r], None, self.iters[r], self.warm, self.stats[t], self.po)

    def outputs(self, t):
        """What the caller of `step(t)`, the latest step, received: the updated state and the step's results, each (rows, S)."""
        r = t % self.ring
        out = {"x": self.x, "xbar": self.xbar, "e": self.e, "status": self.status[r][None], "cost": self.cost[r][None],
               "v": self.v[r], "iters": self.iters[r][None]}
        if self.ablate < 2:
            out["xbar_traj"] = self.traj[r]
        if self.ablate < 1:
            out["tube"] = self.ze1[r]
        return out


DUMP_BYTES = 60_000_000      # --dump-outputs stays below 64 MB: a fixed sample of the scenarios when a step's outputs are larger


def dump_outputs(out_dir, loop, t, s_begin):
    """Writes what step t of `loop` returned as out_dir/<name>.npy in float64, scenarios along the last axis.  When all
    scenarios do not fit in DUMP_BYTES, every array keeps the same seeded sample of them; scenario.npy holds the global
    index of each column.  stats.npy is the step's statistics row, summed with atomics (equal up to summation order)."""
    torch = loop.torch
    os.makedirs(out_dir, exist_ok=True)
    arrays = loop.outputs(t)
    per_scenario = 8 * (1 + sum(a.shape[0] for a in arrays.values()))
    k = min(loop.S, DUMP_BYTES // per_scenario)
    idx = np.arange(loop.S) if k == loop.S else np.sort(np.random.default_rng(0).choice(loop.S, k, replace=False))
    sel = torch.as_tensor(idx, device=loop.dev)
    np.save(os.path.join(out_dir, "scenario.npy"), (s_begin + idx).astype(np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a.index_select(1, sel).cpu().numpy().astype(np.float64))
    np.save(os.path.join(out_dir, "stats.npy"), loop.stats[t].cpu().numpy())


def _nvtx_push(torch, msg):
    try:
        torch.cuda.nvtx.range_push(msg)
    except Exception:      # noqa: BLE001  (NVTX is an annotation, never a reason to fail)
        pass


def _nvtx_pop(torch):
    try:
        torch.cuda.nvtx.range_pop()
    except Exception:      # noqa: BLE001
        pass


def timed_leg(torch, loop, W, K, barrier, use_graph=True, sampler_dev=None):
    """W untimed steps, then K steps in ONE CUDA graph (no host work between steps), CUDA events around the replay.
    Returns (elapsed ms of the K steps, per-step ms list, clocks or None, statistics of the timed steps)."""
    loop.reset(W + K)
    _nvtx_push(torch, f"tzddpc warm-up: {W} closed-loop steps x {loop.S} scenarios")      # (NVTX: visible under nsys / ncu --nvtx)
    for t in range(W):
        loop.step(t)
    _nvtx_pop(torch)
    barrier()
    graph = None
    if use_graph:
        # (no garbage collection inside the capture: a collected controller / ensemble of an earlier leg frees device memory
        #  in its finaliser -- cudaFree -- which invalidates a stream capture in progress)
        gc.collect()
        gc.disable()
        try:
            side = torch.cuda.Stream(device=loop.dev)
            side.wait_stream(torch.cuda.current_stream(loop.dev))
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=side):
                for k in range(K):
                    loop.step(W + k)
        finally:
            gc.enable()
        barrier()
    sampler = ClockSampler(sampler_dev) if sampler_dev is not None else None
    ev = [torch.cuda.Event(enable_timing=True) for _ in range((1 if use_graph else K) + 1)]
    t0 = time.perf_counter()
    _nvtx_push(torch, f"tzddpc timed: {K} closed-loop steps x {loop.S} scenarios")
    ev[0].record()
    if use_graph:
        graph.replay()
        ev[1].record()
    else:
        for k in range(K):
            loop.step(W + k)
            ev[k + 1].record()
    _nvtx_pop(torch)
    if sampler is not None:          # the work is asynchronous: sample the clocks while the GPU goes through it
        while not ev[-1].query():
            sampler.sample()
            time.sleep(0.0005)
    barrier()
    t1 = time.perf_counter()
    elapsed = ev[0].elapsed_time(ev[-1])
    per_step = [elapsed / K] if use_graph else [ev[k].elapsed_time(ev[k + 1]) for k in range(K)]
    clocks = sampler.stop(t0, t1) if sampler else None
    return elapsed, per_step, clocks, loop.stats[W:].clone()


def batch1_latency(tz, ops, torch, dev, steps_per_graph=12, replays=100):
    from tzddpc_b200 import configs
    cfg = configs.double_integrator()
    ctl = build_controller(tz, configs, cfg, dev)
    prog = ctl._program
    n = cfg.n
    g1, nv, N = prog.compiled.g1, prog.compiled.nv, cfg.horizon
    f64 = dict(dtype=torch.float64, device=dev)
    S = 1
    x0 = torch.tensor(cfg.X0[0], **f64)[:, None].contiguous()
    x, xbar, e = x0.clone(), x0.clone(), torch.zeros((n, S), **f64)
    WZ = torch.tensor(np.hstack([cfg.W[0][:, None], cfg.W[1]]), **f64)
    # a random vertex of W per step (examples/1.double_integrator_sim.py:85)
    noise = torch.stack([ops.sample_noise(WZ, S, True, cfg.seed, 0, t) for t in range(steps_per_graph)])
    At, Bt = torch.tensor(cfg.A, **f64), torch.tensor(cfg.B, **f64)
    status = torch.zeros((steps_per_graph, S), dtype=torch.int32, device=dev)
    cost = torch.empty((steps_per_graph, S), **f64)
    v = torch.empty((steps_per_graph, nv, S), **f64)
    traj = torch.empty((steps_per_graph, (N + 1) * n, S), **f64)
    ze1 = torch.empty((steps_per_graph, n * (1 + g1), S), **f64)
    warm = torch.zeros((prog.warm_rows, S), **f64)
    po = tz.SolverOptions(warm_start=2).pack()
    h = prog.handle.value

    def run():
        x.copy_(x0); xbar.copy_(x0); e.zero_(); warm.zero_()      # every replay is the example's 12-step run from X0
        for t in range(steps_per_graph):
            ops.closed_loop_step(h, x, xbar, e, noise[t], x0, At, Bt, status[t], cost[t], v[t], traj[t], ze1[t], None, None, warm,
                                 None, po)

    side = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(side):
        run()                                   # warm-up on the capture stream
    torch.cuda.synchronize(dev)
    graph = torch.cuda.CUDAGraph()
    gc.collect()
    gc.disable()                                # (see timed_leg: no finaliser may free device memory inside a capture)
    try:
        with torch.cuda.graph(graph, stream=side):
            run()
    finally:
        gc.enable()
    for _ in range(3):
        graph.replay()
    torch.cuda.synchronize(dev)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(replays):
        graph.replay()
    b.record()
    torch.cuda.synchronize(dev)
    us = 1e3 * a.elapsed_time(b) / (replays * steps_per_graph)
    # the same through plain launches of the torch op (host in the loop)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for _ in range(4):
        run()
    torch.cuda.synchronize(dev)
    us_eager = 1e6 * (time.perf_counter() - t0) / (4 * steps_per_graph)
    # ... and as ONE launch for the whole run (tz_closed_loop_run: the step loop inside the kernel)
    us_fused, fused_equal = None, None
    if hasattr(ops, "closed_loop_run"):
        ref_x = x.clone()
        status2 = torch.zeros_like(status)
        cost2, v2, traj2, ze2 = torch.empty_like(cost), torch.empty_like(v), torch.empty_like(traj), torch.empty_like(ze1)

        def run_fused():
            x.copy_(x0); xbar.copy_(x0); e.zero_(); warm.zero_()
            ops.closed_loop_run(h, steps_per_graph, x, xbar, e, noise, x0, At, Bt, status2, cost2, v2, traj2, ze2, None, None, None, None, None,
                                warm, None, po)
        run_fused()
        torch.cuda.synchronize(dev)
        fused_equal = bool(torch.equal(x, ref_x) and torch.equal(status2, status) and torch.equal(ze2, ze1))
        g2 = torch.cuda.CUDAGraph()
        gc.collect()
        gc.disable()
        try:
            with torch.cuda.stream(side):
                run_fused()
            torch.cuda.synchronize(dev)
            with torch.cuda.graph(g2, stream=side):
                run_fused()
        finally:
            gc.enable()
        for _ in range(3):
            g2.replay()
        torch.cuda.synchronize(dev)
        a.record()
        for _ in range(replays):
            g2.replay()
        b.record()
        torch.cuda.synchronize(dev)
        us_fused = 1e3 * a.elapsed_time(b) / (replays * steps_per_graph)
    return {"us_per_step": us, "us_per_step_eager_launches": us_eager, "us_per_step_fused_run": us_fused,
            "fused_run_equals_step_loop": fused_equal, "scenarios": 1,
            "workload": "double_integrator: n=2 m=1 T=100 horizon=2 (examples/1.double_integrator_sim.py), closed loop",
            "how": f"CUDA graph of the example's {steps_per_graph} closed-loop steps from X0, {replays} replays, CUDA events",
            "status_ok": bool((status == 0).all().item()), "kernel_bucket": prog.bucket}


def sweep_leg(tz, ops, torch, dev):
    """BASELINE.json configs[1] / BASELINE.md section 1: the double-integrator complexity sweep at batch 1
    (examples/1.double_integrator_computation_complexity.py:48-122): per (method, horizon) the set-up time (identification,
    gain, canonicalisation, program upload -- what the reference's `build_problem` does symbolically) and the latency of the
    first `solve` from X0."""
    from tzddpc_b200 import configs
    cfg = configs.sweep()
    rows = []
    x0 = np.asarray(cfg.X0[0], dtype=np.float64)
    cases = [("tzddpc", N, None) for N in (1, 2, 3, 4, 5)] + [("stzddpc_k0=1", N, 1) for N in (2, 4, 6, 8, 10)] + \
            [("stzddpc_k0=2", N, 2) for N in (3, 5)]
    for name, N, k0 in cases:
        row = {"method": name, "horizon": N}
        try:
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            ctl = build_controller(tz, configs, cfg, dev, horizon=N, k0=k0)
            torch.cuda.synchronize(dev)
            row["setup_s"] = time.perf_counter() - t0
            t0 = time.perf_counter()
            try:
                ctl.solve(x0, np.zeros(cfg.n))
                row["first_solve_status"] = "ok"
            except Exception as exc:      # noqa: BLE001  (the reference raises on an infeasible first step, too)
                row["first_solve_status"] = str(exc)[:60]
            torch.cuda.synchronize(dev)
            row["first_solve_ms"] = 1e3 * (time.perf_counter() - t0)
            t0 = time.perf_counter()
            for _ in range(10):
                try:
                    ctl.solve(x0, np.zeros(cfg.n))
                except Exception:         # noqa: BLE001
                    pass
            row["solve_ms_warm_process"] = 1e2 * (time.perf_counter() - t0)
            row["kernel_bucket"] = ctl._program.bucket
            row["nz"], row["nc"] = ctl._program.compiled.nz, ctl._program.compiled.nc
            row["generators_per_step"] = [int(g) for g in ctl._program.compiled.gens_per_step][:6]
        except Exception as exc:          # noqa: BLE001
            row["error"] = repr(exc)[:160]
        rows.append(row)
    return {"workload": "double-integrator complexity sweep at batch 1 (examples/1.double_integrator_computation_complexity.py)",
            "reference": "BASELINE.md section 1: TZDDPC horizon 1..5 = 5.4 / 6.0 / 12.2 / 70 / 1,623 s per fresh process (build + 1 solve, "
                         "gain synthesis included), 30 GB at horizon 5", "rows": rows}


def datasets_leg(args, tz, ops, torch, dev, cfg, nring):
    """The default workload with the data-set axis: D data sets (seeds cfg.seed + 101 d) of the same plant, one identified
    model / gain / program each (the reference: one TZDDPC object per data set), S / D noise realisations per data set."""
    from tzddpc_b200 import _abi, configs
    D, S = args.datasets, args.scenarios
    per = S // D
    assert per % 16 == 0 and per * D == S, "scenarios must split into D blocks of a multiple of 16"
    n, N = cfg.n, cfg.horizon
    Z = tz.Zonotope
    zon = tz.SystemZonotopes(Z(*cfg.X0), Z(*cfg.U), Z(*cfg.X), Z(*cfg.W))
    f64 = dict(dtype=torch.float64, device=dev)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    # the D data sets are generated on the device (tz_generate_trajectories: examples/utils.py:6-45, one trajectory each) and
    # never leave it; one tz_identify + one tz_gain_synthesis launch for all of them, the host canonicalisation batched over the
    # data sets, one tz_program_create_batch
    zt = lambda c, G: torch.tensor(np.hstack([np.asarray(c, dtype=np.float64)[:, None], np.asarray(G, dtype=np.float64)]), **f64)   # noqa: E731
    Ud, Xd = ops.generate_trajectories(torch.tensor(cfg.A, **f64), torch.tensor(cfg.B, **f64), zt(*cfg.X0), zt(*cfg.U), zt(*cfg.W), D, cfg.T,
                                       cfg.seed, 0)
    torch.cuda.synchronize(dev)
    gen_s = time.perf_counter() - t0
    ens = tz.TZDDPCEnsemble.from_datasets((Ud, Xd), zon, N, tz.StageCost(**cfg.cost),
                                          tz.BoxConstraint(**cfg.box) if cfg.box else tz.BoxConstraint(), scenarios_per_dataset=per,
                                          device=dev)
    torch.cuda.synchronize(dev)
    setup_s = time.perf_counter() - t0
    prog = ens._program
    g1, nv = prog.compiled.g1, prog.compiled.nv
    WZ = torch.tensor(np.hstack([cfg.W[0][:, None], cfg.W[1]]), **f64)
    noise = torch.stack([ops.sample_noise(WZ, S, cfg.noise == "vertex", cfg.seed, 0, t) for t in range(nring)])
    x0 = torch.tensor(cfg.X0[0], **f64)
    x = x0[:, None].repeat(1, S).contiguous()
    xbar, xr, e = x.clone(), x.clone(), torch.zeros((n, S), **f64)
    At, Bt = torch.tensor(cfg.A, **f64), torch.tensor(cfg.B, **f64)
    ze1 = torch.empty((n * (1 + g1), S), **f64)
    traj = torch.empty(((N + 1) * n, S), **f64)
    vbuf, cost = torch.empty((nv, S), **f64), torch.empty(S, **f64)
    status = torch.zeros(S, dtype=torch.int32, device=dev)
    warm = torch.zeros((prog.warm_rows, S), **f64)
    Kd = min(max(args.steps, 20), 100)
    stats = torch.zeros((5 + Kd, _abi.TZ_NSTATS), **f64)
    po = tz.SolverOptions(warm_start=2, check_every=args.check_every, eps_abs=args.eps, eps_rel=args.eps, polish=args.polish).pack()
    h = prog.handle.value

    def step(t):
        ops.closed_loop_step_set(h, x, xbar, e, noise[t % nring], xr, At, Bt, status, cost, vbuf, traj, ze1, None, None, warm,
                                 stats[t], po)

    for t in range(5):
        step(t)
    torch.cuda.synchronize(dev)
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    graph = torch.cuda.CUDAGraph()
    gc.collect()
    gc.disable()                                # (see timed_leg)
    try:
        with torch.cuda.graph(graph, stream=side):
            for k in range(Kd):
                step(5 + k)
    finally:
        gc.enable()
    torch.cuda.synchronize(dev)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    graph.replay()
    b.record()
    torch.cuda.synchronize(dev)
    ms = a.elapsed_time(b) / Kd
    tot = stats[5:].sum(0).cpu().numpy()
    return {"datasets": D, "scenarios_per_dataset": per, "ms_per_step": ms, "value": S / (ms * 1e-3), "unit": UNIT, "steps": Kd,
            "setup_s": setup_s, "setup_generate_data_s": gen_s, "gain": "tz_gain_synthesis (one launch, a robust LQR gain per data set)",
            "gain_iterations_max": int(ens.theta_info["iterations"].max()), "rho_max": float(ens.theta_info["rho"].max()),
            "api": "TZDDPCEnsemble -> tz_closed_loop_step_set (one launch per step, one program per data set)",
            "status_ok_frac": float(1.0 - (tot[3] + tot[4] + tot[6]) / max(tot[7], 1.0)), "iters_mean": float(tot[5] / max(tot[7], 1.0))}


def e2e_legs(args, tz, ops, torch, dev, cfg, prog, loop, K_steps, world, barrier, shard):
    """Host buffers through the C-ABI host entry point: per step the H2D copy of the step's inputs from pinned host memory,
    the fused kernels, and the D2H copy of the step's results, all inside the timed region (wall clock, max over ranks)."""
    from tzddpc_b200 import _abi
    import ctypes as C
    S, n, m, N = loop.S, cfg.n, cfg.m, cfg.horizon
    nv, g1 = prog.compiled.nv, prog.compiled.g1
    nent, nt, nnz = n * (1 + g1), (N + 1) * n, len(prog.tube_pattern)
    Ke = max(3, min(args.e2e_steps, K_steps))
    pin = lambda *shape, dt=torch.float64: torch.empty(shape, dtype=dt).pin_memory()     # noqa: E731
    hx, hxb, he = pin(n, S), pin(n, S), pin(n, S)
    hnoise = pin(Ke + 2, n, S)
    hnoise.copy_(loop.noise[torch.arange(Ke + 2, device=dev) % loop.nring].cpu())
    hcost, hv, htraj, hze = pin(S), pin(nv, S), pin(nt, S), pin(nent, S)
    hu = pin(m, S)
    hstat = pin(S, dt=torch.int32)
    f64 = dict(dtype=torch.float64, device=dev)
    h = prog.handle.value
    L = _abi.lib()
    scratch = torch.zeros(L.tz_closed_loop_step_host_scratch_bytes(h, S) // 8 + 8, **f64)
    Ah, Bh = np.ascontiguousarray(cfg.A), np.ascontiguousarray(cfg.B)
    x0h = pin(n, S)
    x0h.copy_(loop.x0.cpu())

    # chunks of the resident-state call: one GPU 1 / 2 / 4 / 8 chunks = 0.790 / 0.780 / 0.829 / 0.893 ms per step; with several
    # ranks sharing the host's PCIe fabric finer chunks interleave better (2 GPUs: 0.63 ms with 2 chunks, 0.48 with 4)
    nchunks_res = args.e2e_chunks_resident if args.e2e_chunks_resident > 0 else (2 if int(os.environ.get("WORLD_SIZE", "1")) == 1 else 4)

    def leg(packed, resident):
        o_ = ops._opts(tz.SolverOptions(warm_start=int(args.warm_start), check_every=args.check_every, eps_abs=args.eps, eps_rel=args.eps,
                                        polish=args.polish, tube_packed=int(packed), hot_path=int(args.hot_path)).pack())
        hx.copy_(x0h); hxb.copy_(hx); he.zero_()
        scratch.zero_()
        rows = nnz if packed else nent
        if resident:
            # state resident in the caller's device scratch: the first call uploads (x, xbar, e) and x_restart, every later
            # call moves only the step's noise up and (x+, u, cost, status, the packed tube) down
            def host_step(t, first):
                rc = L.tz_closed_loop_run_host(
                    C.c_void_p(h), C.byref(o_), S, 1 if first else 0, C.c_void_p(hx.data_ptr()), C.c_void_p(hxb.data_ptr()),
                    C.c_void_p(he.data_ptr()), C.c_void_p(x0h.data_ptr()), C.c_void_p(hnoise[t].data_ptr()), C.c_void_p(Ah.ctypes.data),
                    C.c_void_p(Bh.ctypes.data), C.c_void_p(hcost.data_ptr()), None, None, C.c_void_p(hze.data_ptr()),
                    C.c_void_p(hu.data_ptr()), C.c_void_p(hstat.data_ptr()), C.c_void_p(scratch.data_ptr()), nchunks_res)
                _abi.check(rc, "tz_closed_loop_run_host")
            h2d = int(n * S * 8 + 8 * (n * n + n * m))
            d2h = int(S * (8 * (n + m + 1 + rows) + 4))
            api = ("tz_closed_loop_run_host (pinned host buffers; x, xbar, e and the active-set hints stay in the caller's device "
                   "scratch between calls; per step: noise up, x+ / u / cost / status / Ze[1].Z down)")
        else:
            def host_step(t, first):
                rc = L.tz_closed_loop_step_host(
                    C.c_void_p(h), C.byref(o_), S, C.c_void_p(hx.data_ptr()), C.c_void_p(hxb.data_ptr()), C.c_void_p(he.data_ptr()),
                    C.c_void_p(hnoise[t].data_ptr()), C.c_void_p(Ah.ctypes.data), C.c_void_p(Bh.ctypes.data),
                    C.c_void_p(hcost.data_ptr()), C.c_void_p(hv.data_ptr()), C.c_void_p(htraj.data_ptr()), C.c_void_p(hze.data_ptr()),
                    C.c_void_p(hstat.data_ptr()), C.c_void_p(scratch.data_ptr()), args.e2e_chunks)
                _abi.check(rc, "tz_closed_loop_step_host")
            h2d = int(4 * n * S * 8 + 8 * (n * n + n * m))
            d2h = int(S * (8 * (3 * n + 1 + nv + nt + rows) + 4))
            api = "tz_closed_loop_step_host (pinned host buffers; every array of the step up and down)"
        for t in range(2):
            host_step(t, t == 0)
        barrier()
        t0 = time.perf_counter()
        for t in range(Ke):
            host_step(2 + t, False)
        barrier()
        dt = shard.max_over_ranks(time.perf_counter() - t0, dev)
        ms = 1e3 * dt / Ke
        return {"value": world * S * Ke / dt, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": Ke,
                "ms_per_step": ms, "h2d_gbs": h2d / (ms * 1e6), "d2h_gbs": d2h / (ms * 1e6), "api": api,
                "tube": (f"packed: {nnz} of {nent} entries of Ze[1].Z per scenario (the others are zero for every "
                         f"(xbar0, e0)); pattern from tz_program_tube_pattern") if packed else "dense n x (1+g1)",
                "solver": "active-set hints carried between calls in the caller's device scratch (warm_start)",
                "status_ok_frac": float((hstat == 0).double().mean().item())}

    out = {}
    has_run = hasattr(L, "tz_closed_loop_run_host")
    out["e2e"] = leg(True, has_run)
    if has_run:
        out["e2e_all_arrays"] = leg(True, False)
    out["e2e_dense_tube"] = leg(False, False)
    return out


def run_stress(args):
    """BASELINE.json configs[4]: synthetic 5-dim system, long horizon, high zonotope order (stress test of the Girard
    reduction), 262,144 scenarios sharded over the GPUs.  Not a reference workload (the reference never reduces Ze); the
    generator spec is fixed here (seed 0).  Two measurements per order cap rho:
      rollout_order*     tz_tube_rollout: product + Minkowski sum + Girard reduction + hull per step with the zonotope resident
                         in shared memory (the fused path; rho <= 30 at n = 5);
      standalone_order*  tz_reach_step / tz_girard_reduce / tz_interval_hull on blocks of the same size: algorithmic bytes (read
                         + written once) over the CUDA-event time, as a fraction of the measured HBM peak;
      chain_order40      the rollout at rho = 40 through the chain of stand-alone kernels (beyond the fused kernel's shared memory).
    `value` = scenario-steps/s of the fused rollout at rho = 20, all ranks."""
    import torch
    import torch.distributed as dist
    from tzddpc_b200 import ops, shard    # noqa: F401  (registers torch.ops.tzddpc.*)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    total = args.scenarios if args.scenarios != 65536 else 262144
    s0, s1 = shard.shard_bounds(total, rank, world)
    S = min(s1 - s0, args.stress_cap) if args.stress_cap > 0 else s1 - s0
    n, m, steps = 5, 1, 32
    rng = np.random.default_rng(0)
    dK = rng.uniform(0.001, 0.02, size=(n, n)); dD = rng.uniform(0.001, 0.02, size=(n, n + m))
    GK = np.zeros((n * n, n, n)); GD = np.zeros((n * (n + m), n, n + m))
    for r in range(n):
        for c in range(n):
            GK[r * n + c, r, c] = dK[r, c]
        for c in range(n + m):
            GD[r * (n + m) + c, r, c] = dD[r, c]
    A = rng.normal(size=(n, n)); A *= 0.85 / np.abs(np.linalg.eigvals(A)).max()
    W = np.hstack([np.zeros((n, 1)), 0.1 * np.ones((n, 1))])
    f = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).to(dev)      # noqa: E731
    peak, peak_src = measured_hbm_peak()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def ev(fn, reps):
        fn()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        barrier()
        return shard.max_over_ranks(a.elapsed_time(b) / reps, dev)

    out = {}
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    for order in (10, 20, 30):
        gcap = n * (order - 1) + n
        Z0 = torch.zeros((S, n, 2), dtype=torch.float64, device=dev)
        Z0[:, :, 0] = torch.rand((S, n), dtype=torch.float64, device=dev, generator=gen) - 0.5
        XU = torch.rand((S, steps, n + m), dtype=torch.float64, device=dev, generator=gen) * 4 - 2
        targs = (f(A), f(GK), f(GD), Z0, XU, f(W), float(order), 0, gcap)
        ms = ev(lambda: torch.ops.tzddpc.tube_rollout(*targs), max(1, args.steps // 10))
        gpre = 26 * gcap + 25 + 30 + 1
        out[f"rollout_order{order}"] = {"ms": ms, "scenario_steps_per_s": world * S * steps / ms * 1e3, "pre_reduce_generators": gpre,
                                        "equiv_unfused_GBps_per_gpu": S * steps * 8 * n * (2 * gpre + 2 * gcap) / ms / 1e6}
        Sz = min(S, 8192)
        Zin = torch.rand((Sz, n, 1 + gcap), dtype=torch.float64, device=dev, generator=gen) - 0.5
        dA_, dGK_ = f(A), f(GK)
        t_reach = ev(lambda: torch.ops.tzddpc.reach_step(dA_, dGK_, Zin, None), 5)
        pre = torch.ops.tzddpc.reach_step(dA_, dGK_, Zin, None)
        b_reach = 8 * n * Sz * ((1 + gcap) + pre.shape[2])
        t_gir = ev(lambda: torch.ops.tzddpc.girard_reduce(pre, float(order), 0, gcap), 5)
        b_gir = 8 * n * Sz * (pre.shape[2] + 1 + gcap)
        t_hull = ev(lambda: torch.ops.tzddpc.interval_hull(pre), 5)
        b_hull = 8 * n * Sz * pre.shape[2]
        out[f"standalone_order{order}"] = {"frac_reach": b_reach / t_reach / 1e6 / peak, "frac_girard": b_gir / t_gir / 1e6 / peak,
                                           "frac_hull": b_hull / t_hull / 1e6 / peak, "girard_GBps": b_gir / t_gir / 1e6,
                                           "generators_in": int(pre.shape[2] - 1), "zonotopes_per_gpu": Sz}
        del Z0, XU, Zin, pre
    # ---- order 40 (configs[4] names rho = 10..40): the fused rollout keeps the pre-reduction block in shared memory and stops
    # at order 30 for n = 5 (order 40 needs 278 KB); beyond that the same recursion runs through the chain of stand-alone
    # kernels -- tz_reach_step (M_K x Ze and M_Delta x (x, u) + W), concatenation, tz_girard_reduce, tz_interval_hull per step
    order = 40
    gcap = n * (order - 1) + n
    Sc = min(S, 4096)
    Z0 = torch.zeros((Sc, n, 2), dtype=torch.float64, device=dev)
    Z0[:, :, 0] = torch.rand((Sc, n), dtype=torch.float64, device=dev, generator=gen) - 0.5
    XU = torch.rand((Sc, steps, n + m), dtype=torch.float64, device=dev, generator=gen) * 4 - 2
    dA_, dGK_, dGD_, dW_ = f(A), f(GK), f(GD), f(W)
    zeroC = torch.zeros((n, n + m), dtype=torch.float64, device=dev)
    state = {}

    def chain():
        Z = Z0
        for k in range(steps):
            T1 = torch.ops.tzddpc.reach_step(dA_, dGK_, Z, None)
            xu = torch.zeros((Sc, n + m, 2), dtype=torch.float64, device=dev)
            xu[:, :, 0] = XU[:, k]
            Zn = torch.ops.tzddpc.reach_step(zeroC, dGD_, xu, dW_)
            pre = torch.cat([T1, Zn[:, :, 1:]], dim=2)
            pre[:, :, 0] += Zn[:, :, 0]
            red, gout = torch.ops.tzddpc.girard_reduce(pre, float(order), 0, gcap)
            Z = red
            lo, hi = torch.ops.tzddpc.interval_hull(Z)
        state["gmax"], state["width"] = gout, hi - lo

    ms = ev(chain, 1)
    out["chain_order40"] = {"ms": ms, "scenario_steps_per_s": world * Sc * steps / ms * 1e3, "scenarios_per_gpu": Sc,
                            "generators_after_reduction": int(state["gmax"].max().item()), "pre_reduce_generators": 26 * gcap + 25 + 30 + 1,
                            "mean_tube_width_last_step": float(state["width"].mean().item()),
                            "how": "reach_step x2 + cat + girard_reduce + interval_hull per step (stand-alone kernels; the fused rollout "
                                   "stops at order 30)"}
    del Z0, XU
    r20 = out["rollout_order20"]
    line = {"metric": "tube-rollout scenario-steps/s (synthetic stress: Girard order cap 20, horizon 32)", "value": r20["scenario_steps_per_s"],
            "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r20["ms"] / steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"stress: synthetic 5-dim system, horizon {steps}, Girard order cap 10 / 20 / 30, {world * S} scenarios over "
                                   f"{world} GPU(s) (BASELINE.json configs[4]: 262,144 over 8)", "scenarios_this_rank": S,
                       "parallelism": f"scenario-dp{world}"},
            "gpu_launches": 3 * (1 + max(1, args.steps // 10)), "roofline": {"bound": "hbm", "peak": peak, "unit": "GB/s", "peak_source": peak_src,
                                                                            "achieved": out["standalone_order20"]["girard_GBps"],
                                                                            "frac": out["standalone_order20"]["frac_girard"],
                                                                            "kernel": "tz::girard_kernel", "traffic": None},
            "stress": out}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_gpu(args):
    import torch
    import torch.distributed as dist
    import tzddpc_b200 as tz
    from tzddpc_b200 import configs, ops, shard

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg = configs.CONFIGS[args.workload]()
    K_steps, W_steps = args.steps, args.warmup
    n, m, N = cfg.n, cfg.m, cfg.horizon
    S_total = total_scenarios(args, world)
    s_begin, s_end = shard.shard_bounds(S_total, rank, world)
    S = s_end - s_begin
    if args.scaling == "strong":
        assert S_total % (16 * world) == 0, "the shards must be whole 16-scenario tiles"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    ctl = build_controller(tz, configs, cfg, dev)
    prog = ctl._program
    g1 = prog.compiled.g1
    nnz = len(prog.tube_pattern)

    def mk_opts(packed):
        return tz.SolverOptions(warm_start=int(args.warm_start), check_every=args.check_every, eps_abs=args.eps, eps_rel=args.eps,
                                polish=args.polish, hot_path=int(args.hot_path), tube_packed=int(packed))

    total = W_steps + K_steps
    nring = min(max(total, 8), 64)
    dense = ClosedLoop(tz, ops, torch, ctl, cfg, dev, S, s_begin, nring, mk_opts(args.packed), seed=cfg.seed, ablate=args.ablate)
    use_graph = not args.no_graph and not args.dump_steps
    hot = bool(args.hot_path) and int(args.warm_start) == 2 and prog.bucket.startswith("B0")
    launches_per_step = 2 if hot else 1

    # ---- headline: dense tube, state resident in HBM
    elapsed_ms, kern_ms, clocks, stats = timed_leg(torch, dense, W_steps, K_steps, barrier, use_graph, local if rank == 0 else None)
    elapsed_ms = shard.max_over_ranks(elapsed_ms, dev)
    tot_stats = shard.reduce_statistics(stats.clone()).sum(0).cpu().numpy()
    cnt = max(tot_stats[7], 1.0)
    if args.dump_steps and rank == 0:
        np.savez(args.dump_steps, kern_ms=np.asarray(kern_ms), stats=stats.cpu().numpy())
    if args.dump_outputs and rank == 0:          # before any later leg reuses `dense`
        dump_outputs(args.dump_outputs, dense, W_steps + K_steps - 1, s_begin)
    value = S_total * K_steps / (elapsed_ms * 1e-3)
    rows_headline = nnz if args.packed else n * (1 + g1)
    bstep = algorithmic_bytes_per_scenario_step(n, m, N, g1, rows_headline)
    peak, peak_src = measured_hbm_peak()
    avg_kernel_ms = float(np.mean(kern_ms))
    achieved = bstep * S / (avg_kernel_ms * 1e-3) / 1e9
    kname = "tz::fast_step_kernel" if hot else "tz::step_kernel"
    ev_ncu = ncu_evidence(kname + ("/packed" if args.packed else "/dense")) or {}
    l2note = (" > 126 MB L2 (inputs larger than L2)" if bstep * S > 126e6 else
              "; a ring of 4 output buffers is cycled, the per-step inputs are the previous step's outputs")
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K_steps, "warmup": W_steps,
            "ms_per_step": elapsed_ms / K_steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(cfg, S_total, world, args.scaling), "scenarios_total": S_total, "scenarios_this_rank": S,
                       "parallelism": f"scenario-dp{world}",
                       "l2": f"per-step HBM traffic {bstep * S / 1e6:.0f} MB per GPU" + l2note,
                       "solver": {"warm_start": {0: "cold", 1: "previous (x, y)", 2: "active-set hint of the previous step (KKT-certified)"}[int(args.warm_start)],
                                  "hot_path": ("fast_step_kernel (closed-form certificate, one thread per scenario) + step_kernel on the deferred tiles"
                                               if hot else "step_kernel (ADMM lane groups)"),
                                  "eps": args.eps, "certificate": "active-set KKT"},
                       "kernel_bucket": prog.bucket, "tube": "packed" if args.packed else "dense n x (1+g1)",
                       "episodes": "a scenario whose step is infeasible (the reference raises: end of that run) starts a new "
                                   "run from x0; the 5-dim example reaches that point every ~62 steps (DESIGN.md section 6, "
                                   "tests/golden/ex3_sensitivity.json)",
                       "noise": f"Philox4x32-10 keyed by (seed, global scenario, t): {nring} realisations per scenario, cycled"},
            "gpu_launches": K_steps * launches_per_step, "launch_mode": "one CUDA graph of the K steps" if use_graph else "eager",
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": ev_ncu.get("dram_bytes_per_launch"), "peak_source": peak_src, "bytes_per_scenario_step": bstep,
                         "kernel_ms_avg": avg_kernel_ms, "kernel": kname,
                         "fp64_fraction": ev_ncu.get("fp64_pipe_frac"), "issue_fraction": ev_ncu.get("issue_active_frac"),
                         "ncu_source": ev_ncu.get("source")},
            "solver_stats": {"iters_mean": float(tot_stats[5] / cnt), "iters_max_last_steps": int(dense.iters.max().item()),
                             "status_ok_frac": float(1.0 - (tot_stats[3] + tot_stats[4] + tot_stats[6]) / cnt),
                             "infeasible": int(tot_stats[3]), "maxiter": int(tot_stats[4]), "nonfinite": int(tot_stats[6]),
                             "mean_norm_x": float(tot_stats[0] / cnt)},
            "clocks": clocks}

    # ---- shard invariance (strong scaling): the shards' final states, gathered, equal the single-GPU run bit for bit
    if world > 1 and args.scaling == "strong" and not args.no_invariance:
        gathered = [torch.empty((n, S), dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(gathered, dense.x.contiguous())
        if rank == 0:
            full = ClosedLoop(tz, ops, torch, ctl, cfg, dev, S_total, 0, nring, mk_opts(args.packed), seed=cfg.seed)
            full.reset(total)
            for t in range(total):
                full.step(t)
            torch.cuda.synchronize(dev)
            got = torch.cat(gathered, dim=1)
            line["shard_invariance"] = {"bitwise_equal_final_state": bool(torch.equal(got, full.x)), "steps": total, "scenarios": S_total,
                                        "how": "all_gather of the shards' x after the timed steps vs the same closed loop on rank 0 alone"}
            del full
        barrier()

    if not args.quick:
        # ---- the packed tube: what the kernels do when the structural zeros of Ze[1].Z are not written
        packed = ClosedLoop(tz, ops, torch, ctl, cfg, dev, S, s_begin, nring, mk_opts(1), seed=cfg.seed)
        el_p, k_p, _, _ = timed_leg(torch, packed, W_steps, K_steps, barrier, use_graph)
        el_p = shard.max_over_ranks(el_p, dev)
        bp = algorithmic_bytes_per_scenario_step(n, m, N, g1, nnz)
        ev_p = ncu_evidence(kname + "/packed") or {}
        ach_p = bp * S / (float(np.mean(k_p)) * 1e-3) / 1e9
        line["roofline_packed"] = {"bound": "hbm", "achieved": ach_p, "peak": peak, "unit": "GB/s", "frac": ach_p / peak,
                                   "bytes_per_scenario_step": bp, "kernel_ms_avg": float(np.mean(k_p)), "ms_per_step": el_p / K_steps,
                                   "value": S_total * K_steps / (el_p * 1e-3), "traffic": ev_p.get("dram_bytes_per_launch"),
                                   "fp64_fraction": ev_p.get("fp64_pipe_frac"), "issue_fraction": ev_p.get("issue_active_frac"),
                                   "note": f"{nnz} of {n * (1 + g1)} tube entries per scenario: the step is bound by FP64 issue / latency, not by HBM"}
        del packed
        # ---- regimes: the driver's window ends before the first infeasibility wave (step ~62 of the 5-dim example); a 200-step
        # window contains three of them (restarts from the run-start hint)
        if K_steps < 150 and args.regime_steps > 0:
            el_r, _, _, st_r = timed_leg(torch, dense, W_steps, args.regime_steps, barrier, use_graph)
            el_r = shard.max_over_ranks(el_r, dev)
            tr = shard.reduce_statistics(st_r.clone()).sum(0).cpu().numpy()
            line["regimes"] = {f"steps_{W_steps}_{W_steps + K_steps}": {"ms_per_step": elapsed_ms / K_steps, "infeasible_frac": float(tot_stats[3] / cnt)},
                               f"steps_{W_steps}_{W_steps + args.regime_steps}": {"ms_per_step": el_r / args.regime_steps,
                                                                                 "infeasible_frac": float(tr[3] / max(tr[7], 1.0)),
                                                                                 "iters_mean": float(tr[5] / max(tr[7], 1.0))}}
        # ---- weak scaling beside the strong headline
        if world > 1 and args.scaling == "strong":
            wl = ClosedLoop(tz, ops, torch, ctl, cfg, dev, S_total, rank * S_total, nring, mk_opts(args.packed), seed=cfg.seed)
            el_w, _, _, _ = timed_leg(torch, wl, W_steps, K_steps, barrier, use_graph)
            el_w = shard.max_over_ranks(el_w, dev)
            line["weak_scaling"] = {"scenarios_per_gpu": S_total, "ms_per_step": el_w / K_steps,
                                    "value": world * S_total * K_steps / (el_w * 1e-3), "unit": UNIT}
            del wl

    # ---- e2e
    if not args.no_e2e:
        line.update(e2e_legs(args, tz, ops, torch, dev, cfg, prog, dense, K_steps, world, barrier, shard))

    single = rank == 0 and world == 1 and not args.quick
    # ---- data-set axis (north_star: scenarios = noise realisations x initial states x data sets): D data sets, one
    # program each, the whole batch in one launch per step (tz_closed_loop_step_set); rank 0 at N = 1 only
    if single and args.datasets > 0:
        try:
            line["datasets_axis"] = datasets_leg(args, tz, ops, torch, dev, cfg, nring)
        except Exception as exc:      # noqa: BLE001  (secondary leg: never fail the headline line)
            line["datasets_axis"] = {"error": repr(exc)[:300]}
    # ---- the other BASELINE.json configs, driver-visible (rank 0, N = 1): configs[0] batch-1 latency, configs[1] the sweep,
    # configs[2] the pulley with 4,096 scenarios
    if single and not args.no_batch1:
        try:
            line["batch1"] = batch1_latency(tz, ops, torch, dev)
        except Exception as exc:      # noqa: BLE001
            line["batch1"] = {"error": repr(exc)[:200]}
    if single and not args.no_other_configs:
        try:
            pc = configs.pulley()
            pctl = build_controller(tz, configs, pc, dev)
            pl = ClosedLoop(tz, ops, torch, pctl, pc, dev, 4096, 0, 64, mk_opts(0), seed=pc.seed)
            el, _, _, st = timed_leg(torch, pl, 5, 200, barrier, True)
            ts = st.sum(0).cpu().numpy()
            pb = algorithmic_bytes_per_scenario_step(pc.n, pc.m, pc.horizon, pctl._program.compiled.g1)
            line["pulley_4096"] = {"workload": "examples/2.pulley_sim.py: n=4 m=1 T=400 horizon=2, 4,096 noise realisations, 200 steps "
                                               "(BASELINE.json configs[2])",
                                   "ms_per_step": el / 200, "value": 4096 * 200 / (el * 1e-3), "unit": UNIT,
                                   "status_ok_frac": float(1.0 - (ts[3] + ts[4] + ts[6]) / max(ts[7], 1.0)),
                                   "iters_mean": float(ts[5] / max(ts[7], 1.0)), "hbm_frac": pb * 4096 / (el / 200 * 1e-3) / 1e9 / peak,
                                   "reference": "BASELINE.md: 5 runs x 200 steps in 8.4-13.1 s each (~55 ms per step, one scenario)"}
            del pl, pctl
        except Exception as exc:      # noqa: BLE001
            line["pulley_4096"] = {"error": repr(exc)[:200]}
        try:
            line["sweep"] = sweep_leg(tz, ops, torch, dev)
        except Exception as exc:      # noqa: BLE001
            line["sweep"] = {"error": repr(exc)[:200]}

    # ---- CPU baseline on this box's host cores (rank 0, N = 1 only): the oracle port, one process per core, on the window
    # of the closed loop the GPU leg timed (steps W .. W+K), `--cpu-scen` scenarios per core
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = len(os.sched_getaffinity(0)) if args.cpu_cores <= 0 else args.cpu_cores
        val, secs = cpu_oracle_throughput(args.workload, cores, args.cpu_scen, W_steps, K_steps)
        line["cpu_baseline"] = {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": f"{cores * args.cpu_scen} scenarios ({args.cpu_scen} per core) x steps {W_steps}..{W_steps + K_steps} of the "
                                          f"closed loop ({secs:.1f} s), numpy oracle of the reference path (same code path as --impl reference)",
                                "per_core": val / cores}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="fivedim", choices=["fivedim", "pulley", "double_integrator", "stress"])
    ap.add_argument("--stress-cap", type=int, default=0, help="stress workload: cap on the scenarios per GPU (0 = the whole shard)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong: --scenarios in total, sharded over the GPUs (BASELINE.json configs[3]); weak: --scenarios per GPU")
    ap.add_argument("--scenarios", type=int, default=65536)
    ap.add_argument("--warm-start", type=int, default=2, help="0 cold, 1 previous (x, y), 2 active-set hint (default)")
    ap.add_argument("--check-every", type=int, default=8)
    ap.add_argument("--eps", type=float, default=1e-6)
    ap.add_argument("--polish", type=int, default=3, help="augmented-Lagrangian iterations of the certificate / polish")
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--e2e-chunks", type=int, default=2)
    ap.add_argument("--e2e-chunks-resident", type=int, default=0, help="chunks of the resident-state host call (0: 2 on one GPU, 4 per rank on several)")
    ap.add_argument("--regime-steps", type=int, default=200, help="length of the long window of the `regimes` leg (0 = skip)")
    ap.add_argument("--datasets", type=int, default=4096, help="data sets of the data-set-axis leg (0 = skip)")
    ap.add_argument("--cpu-scen", type=int, default=48, help="scenarios per core of the CPU baseline")
    ap.add_argument("--cpu-cores", type=int, default=0, help="processes of the CPU baseline (0 = all host cores)")
    ap.add_argument("--dump-steps", default="", help="write per-step kernel ms and solver statistics to this .npz (diagnostics)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (float64, under 64 MB; rank 0's shard)")
    ap.add_argument("--ablate", type=int, default=0, help="diagnostics only: 1 = do not write Ze[1].Z, 2 = nor the trajectory")
    ap.add_argument("--hot-path", type=int, default=1, help="0: the ADMM kernel for every tile (diagnostics)")
    ap.add_argument("--packed", type=int, default=0, help="1: packed tube in the device-timed headline leg (diagnostics)")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches instead of one CUDA graph of the K steps")
    ap.add_argument("--quick", action="store_true", help="headline (+ e2e / cpu unless disabled) only: no secondary legs")
    ap.add_argument("--no-batch1", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--no-invariance", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload == "stress"):
        ap.error("--dump-outputs writes the native closed-loop step; it has no meaning for --impl reference or --workload stress")
    if args.warmup < 3:
        args.warmup = 3
    if args.workload == "stress":
        if args.impl == "reference":
            print(json.dumps({"impl": "reference", "unavailable": "the stress configuration is not a reference workload (the reference never reduces Ze)"}))
        else:
            run_stress(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
