#!/usr/bin/env python
"""Closed loop of a program set (the data-set axis, TZDDPCEnsemble) as a step loop -- one tz_closed_loop_step_set launch per
step -- against the fused run -- tz_closed_loop_run_set, the whole run in one launch -- in one process:

    python profiles/ensemble_run.py [--datasets 1,2,4,8,15,64] [--per 16] [--steps 12,200] [--rounds 5] [--out FILE]

5-dim example (examples/3.5dimsystem_sim.py), one controller per data set (16 distinct data sets, cycled beyond 16), `per`
scenarios each, warm_start = 2 (active-set hints).  Each variant is a CUDA graph of one run of K steps restarted from X0 on
every replay; CUDA events time the replays.  The two variants are timed in turn, `rounds` times, so that drift on a shared
machine hits them alike.  Both runs are compared after the warm-up: final state and the status of every step bit-equal,
cost and input of every successful step bit-equal.  Prints one JSON object (and writes it to --out): the card, its power limit, and µs per step of every round,
variant and size."""
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


def controllers(cfg, D):
    ctls = []
    Z = tz.Zonotope
    zon = tz.SystemZonotopes(Z(*cfg.X0), Z(*cfg.U), Z(*cfg.X), Z(*cfg.W))
    for d in range(D):
        u, x = configs.generate_dataset(cfg, np.random.default_rng(cfg.seed + 101 * d))
        t = tz.TZDDPC(tz.Data(u, x))
        t.verbose = False
        t.build_zonotopes(zon)
        C = t.Mdata.center
        t.build_zonotopes_theta(zon, K=configs.lqr_gain(C[:, :cfg.n], C[:, cfg.n:]))
        t.build_problem(cfg.horizon, tz.StageCost(**cfg.cost), tz.BoxConstraint(**cfg.box))
        ctls.append(t)
    return ctls


def capture(fn, side, dev):
    with torch.cuda.stream(side):
        fn()                                    # warm-up on the capture stream
    torch.cuda.synchronize(dev)
    g = torch.cuda.CUDAGraph()
    gc.collect()
    gc.disable()                                # (no finaliser may free device memory inside a capture)
    try:
        with torch.cuda.graph(g, stream=side):
            fn()
    finally:
        gc.enable()
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize(dev)
    return g


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--datasets", default="1,2,4,8,15,64")
    ap.add_argument("--per", type=int, default=16)
    ap.add_argument("--steps", default="12,200")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--step-budget", type=int, default=2400, help="closed-loop steps per timed window (replays x K)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    sizes = [int(v) for v in args.datasets.split(",")]
    step_counts = [int(v) for v in args.steps.split(",")]
    cfg = configs.fivedim()
    base = controllers(cfg, min(16, max(sizes)))
    dev = base[0].device
    f64 = dict(dtype=torch.float64, device=dev)
    n, m, N = cfg.n, cfg.m, cfg.horizon
    At, Bt = torch.tensor(cfg.A, **f64), torch.tensor(np.asarray(cfg.B).reshape(n, m), **f64)
    WZ = base[0]._t(base[0].zonotopes.W.Z)
    po = tz.SolverOptions(warm_start=2).pack()
    side = torch.cuda.Stream(device=dev)
    results = []
    for D in sizes:
        ens = tz.TZDDPCEnsemble([base[d % len(base)] for d in range(D)], args.per)
        S, h = ens.num_scenarios, ens._program.handle.value
        nv = ens._dims[1]
        for K in step_counts:
            noise = torch.stack([ops.sample_noise(WZ, S, False, 3, 0, k) for k in range(K)])
            x0 = ens._t(np.tile(cfg.X0[0], (S, 1)).T)
            bufs = {}
            for var in ("loop", "fused"):
                bufs[var] = dict(x=x0.clone(), xbar=x0.clone(), e=torch.zeros((n, S), **f64),
                                 status=torch.zeros((K, S), dtype=torch.int32, device=dev), cost=torch.empty((K, S), **f64),
                                 v=torch.empty((K, nv, S), **f64), u=torch.empty((K, m, S), **f64),
                                 warm=torch.zeros((ens._program.warm_rows, S), **f64))

            def loop(b=bufs["loop"]):
                b["x"].copy_(x0); b["xbar"].copy_(x0); b["e"].zero_(); b["warm"].zero_()
                for k in range(K):
                    ops.closed_loop_step_set(h, b["x"], b["xbar"], b["e"], noise[k], x0, At, Bt, b["status"][k], b["cost"][k], b["v"][k],
                                             None, None, b["u"][k], None, b["warm"], None, po)

            def fused(b=bufs["fused"]):
                b["x"].copy_(x0); b["xbar"].copy_(x0); b["e"].zero_(); b["warm"].zero_()
                ops.closed_loop_run_set(h, K, b["x"], b["xbar"], b["e"], noise, x0, At, Bt, b["status"], b["cost"], b["v"], None, None,
                                        b["u"], None, None, None, None, b["warm"], None, po)

            graphs = {"loop": capture(loop, side, dev), "fused": capture(fused, side, dev)}
            a_, b_ = bufs["loop"], bufs["fused"]
            good = a_["status"] == 0           # (values of failed steps: see tests/test_gpu_fused_run.py)
            equal = all(torch.equal(a_[k], b_[k]) for k in ("x", "xbar", "e", "status")) and \
                torch.equal(a_["cost"][good], b_["cost"][good]) and \
                torch.equal(a_["u"].permute(0, 2, 1)[good], b_["u"].permute(0, 2, 1)[good])
            replays = max(1, args.step_budget // K)
            us = {"loop": [], "fused": []}
            for _ in range(args.rounds):
                for var in ("loop", "fused"):
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    for _ in range(replays):
                        graphs[var].replay()
                    b.record()
                    torch.cuda.synchronize(dev)
                    us[var].append(1e3 * a.elapsed_time(b) / (replays * K))
            med = {k: float(np.median(v)) for k, v in us.items()}
            results.append({"datasets": D, "scenarios": S, "steps": K, "replays": replays, "bit_equal": bool(equal),
                            "infeasible_share": float((a_["status"] == 2).double().mean().item()),
                            "us_per_step": {k: [round(q, 3) for q in v] for k, v in us.items()},
                            "median_us_per_step": {k: round(v, 3) for k, v in med.items()},
                            "spread_us_per_step": {k: round(float(np.max(v) - np.min(v)), 3) for k, v in us.items()},
                            "loop_over_fused": round(med["loop"] / med["fused"], 3)})
            print(json.dumps(results[-1]), file=sys.stderr, flush=True)
            del graphs
            torch.cuda.synchronize(dev)
    out = {"card": card(), "example": "fivedim", "scenarios_per_dataset": args.per, "options": "warm_start=2",
           "timing": "CUDA events around CUDA-graph replays of one K-step run from X0; loop and fused alternated per round",
           "results": results}
    text = json.dumps(out)
    print(text)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
