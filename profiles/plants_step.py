#!/usr/bin/env python
"""Step time of the 5-dim closed loop with a plant per scenario (tz_closed_loop_step_plants, plants drawn from M_Sigma by
tz_sample_plants) against the shared plant (tz_closed_loop_step), dense and packed tube, in one process:

    python profiles/plants_step.py [--scenarios 65536] [--steps 8] [--replays 20] [--rounds 5]

Each variant is a CUDA graph of `steps` closed-loop steps (warm_start = 2, the hot path) restarted from X0 on every replay;
CUDA events time `replays` replays.  The four variants are timed in turn, `rounds` times, so that drift on a shared machine
hits them alike.  Prints one JSON object: the card, its power limit, ms per step of every round and variant, and the
algorithmic bytes per scenario-step (SURVEY.md 8d, + 8 n(n+m) for the plant)."""
import argparse
import gc
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import tzddpc_b200 as tz  # noqa: E402
from tzddpc_b200 import configs, ops  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenarios", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--replays", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    cfg = configs.fivedim()
    u, x = configs.generate_dataset(cfg, np.random.default_rng(cfg.seed))
    t = tz.TZDDPC(tz.Data(u, x))
    t.verbose = False
    Z = tz.Zonotope
    zon = tz.SystemZonotopes(Z(*cfg.X0), Z(*cfg.U), Z(*cfg.X), Z(*cfg.W))
    t.build_zonotopes(zon)
    C = t.Mdata.center
    t.build_zonotopes_theta(zon, K=configs.lqr_gain(C[:, :cfg.n], C[:, cfg.n:]))
    t.build_problem(cfg.horizon, tz.StageCost(**cfg.cost), tz.BoxConstraint(**cfg.box))
    S, K, n, m = args.scenarios, args.steps, cfg.n, cfg.m
    dev = t.device
    f64 = dict(dtype=torch.float64, device=dev)
    prog = t._program
    nv, g1, N = prog.compiled.nv, prog.compiled.g1, cfg.horizon
    A, B = t.sample_plants(S, seed=7)
    AB = torch.cat([A, B], dim=2).reshape(S, -1).t().contiguous()
    At, Bt = torch.tensor(cfg.A, **f64), torch.tensor(cfg.B, **f64)
    WZ = t._t(t.zonotopes.W.Z)
    noise = torch.stack([ops.sample_noise(WZ, S, False, 3, 0, k) for k in range(K)])
    x0 = t._t(np.tile(cfg.X0[0], (S, 1)).T)
    x, xbar, e = x0.clone(), x0.clone(), torch.zeros((n, S), **f64)
    status = torch.zeros((K, S), dtype=torch.int32, device=dev)
    cost, v, traj = torch.empty((K, S), **f64), torch.empty((K, nv, S), **f64), torch.empty((K, (N + 1) * n, S), **f64)
    rows = {0: n * (1 + g1), 1: len(prog.tube_pattern)}
    ze1 = {p: torch.empty((K, r, S), **f64) for p, r in rows.items()}
    warm = torch.zeros((prog.warm_rows, S), **f64)
    h = prog.handle.value

    def run(plants, packed):
        po = tz.SolverOptions(warm_start=2, tube_packed=packed).pack()
        x.copy_(x0); xbar.copy_(x0); e.zero_(); warm.zero_()
        for k in range(K):
            if plants:
                ops.closed_loop_step_plants(h, x, xbar, e, noise[k], x0, AB, status[k], cost[k], v[k], traj[k], ze1[packed][k], None, None,
                                            warm, None, po)
            else:
                ops.closed_loop_step(h, x, xbar, e, noise[k], x0, At, Bt, status[k], cost[k], v[k], traj[k], ze1[packed][k], None, None,
                                     warm, None, po)

    variants = [(pl, pk) for pk in (0, 1) for pl in (False, True)]
    side = torch.cuda.Stream(device=dev)
    graphs = {}
    for var in variants:
        with torch.cuda.stream(side):
            run(*var)
        torch.cuda.synchronize(dev)
        g = torch.cuda.CUDAGraph()
        gc.collect()
        gc.disable()
        try:
            with torch.cuda.graph(g, stream=side):
                run(*var)
        finally:
            gc.enable()
        for _ in range(3):
            g.replay()
        graphs[var] = g
    torch.cuda.synchronize(dev)
    ms = {var: [] for var in variants}
    infeasible = {}
    for _ in range(args.rounds):
        for var in variants:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(args.replays):
                graphs[var].replay()
            b.record()
            torch.cuda.synchronize(dev)
            ms[var].append(a.elapsed_time(b) / (args.replays * K))
            infeasible[var] = float((status == 2).double().mean().item())
    name = lambda var: ("plants" if var[0] else "shared") + ("_packed" if var[1] else "_dense")       # noqa: E731
    base = 8 * (6 * n + N * m + (N + 1) * n + 1) + 4
    out = {"card": card(), "scenarios": S, "steps_per_graph": K, "replays": args.replays,
           "ms_per_step": {name(v_): [round(q, 5) for q in ms[v_]] for v_ in variants},
           "median_ms_per_step": {name(v_): round(float(np.median(ms[v_])), 5) for v_ in variants},
           "infeasible_share": {name(v_): infeasible[v_] for v_ in variants},
           "bytes_per_scenario_step": {"shared_dense": base + 8 * rows[0], "shared_packed": base + 8 * rows[1],
                                       "plants_dense": base + 8 * rows[0] + 8 * n * (n + m),
                                       "plants_packed": base + 8 * rows[1] + 8 * n * (n + m)}}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
