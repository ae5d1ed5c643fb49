#!/usr/bin/env python
"""The fused tube rollout (tz_tube_rollout) across Girard order caps, with the pre-reduction block resident in shared memory
(tube_rollout_kernel) and recomputed (tube_rollout_recompute_kernel), on the stress workload of bench.py (BASELINE.json
configs[4]: synthetic 5-dim system, generator spec of seed 0, horizon 32), in one process:

    python profiles/rollout_orders.py [--scenarios 262144] [--chain-scenarios 4096] [--rounds 3]

  full size:  resident and recompute at orders 10 / 20 / 30, recompute at 40 / 60, `--scenarios` scenarios;
  order 40:   recompute against the chain of stand-alone kernels exactly as bench.py's chain_order40 runs it
              (reach_step x2 + cat + girard_reduce + interval_hull per step), `--chain-scenarios` scenarios.
TZDDPC_ROLLOUT selects the kernel per launch.  CUDA events time each variant, the variants are timed in turn, `rounds`
times, so that drift on a shared machine hits them alike.  Prints one JSON object: the card, its power limit, ms per
rollout of every round and variant, the median and the spread (max / min - 1) and the median scenario-steps/s."""
import argparse
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from tzddpc_b200 import ops  # noqa: E402,F401  (registers torch.ops.tzddpc.*)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenarios", type=int, default=262144)
    ap.add_argument("--chain-scenarios", type=int, default=4096)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    dev = torch.device("cuda")
    n, m, steps = 5, 1, 32
    rng = np.random.default_rng(0)                 # bench.py run_stress
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
    dA, dGK, dGD, dW = f(A), f(GK), f(GD), f(W)
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234)

    def inputs(S):
        Z0 = torch.zeros((S, n, 2), dtype=torch.float64, device=dev)
        Z0[:, :, 0] = torch.rand((S, n), dtype=torch.float64, device=dev, generator=gen) - 0.5
        XU = torch.rand((S, steps, n + m), dtype=torch.float64, device=dev, generator=gen) * 4 - 2
        return Z0, XU

    def rollout(kernel, order, Z0, XU):
        def run():
            os.environ["TZDDPC_ROLLOUT"] = kernel
            return torch.ops.tzddpc.tube_rollout(dA, dGK, dGD, Z0, XU, dW, float(order), 0, n * (order - 1) + n)
        return run

    def chain(order, Z0, XU):
        Sc, gcap = Z0.shape[0], n * (order - 1) + n
        zeroC = torch.zeros((n, n + m), dtype=torch.float64, device=dev)

        def run():
            os.environ.pop("TZDDPC_ROLLOUT", None)
            Z = Z0
            for k in range(steps):
                T1 = torch.ops.tzddpc.reach_step(dA, dGK, Z, None)
                xu = torch.zeros((Sc, n + m, 2), dtype=torch.float64, device=dev)
                xu[:, :, 0] = XU[:, k]
                Zn = torch.ops.tzddpc.reach_step(zeroC, dGD, xu, dW)
                pre = torch.cat([T1, Zn[:, :, 1:]], dim=2)
                pre[:, :, 0] += Zn[:, :, 0]
                Z, gout = torch.ops.tzddpc.girard_reduce(pre, float(order), 0, gcap)
                lo, hi = torch.ops.tzddpc.interval_hull(Z)
            return Z, gout, lo, hi
        return run

    S, Sc = args.scenarios, args.chain_scenarios
    full = inputs(S)
    small = inputs(Sc)
    variants = {}                                  # name -> (fn, scenarios, launches per timing)
    for order in (10, 20, 30):
        for kernel in ("resident", "recompute"):
            variants[f"{kernel}_order{order}"] = (rollout(kernel, order, *full), S, 1)
    for order in (40, 60):
        variants[f"recompute_order{order}"] = (rollout("recompute", order, *full), S, 1)
    variants[f"recompute_order40_S{Sc}"] = (rollout("recompute", 40, *small), Sc, 10)
    variants[f"chain_order40_S{Sc}"] = (chain(40, *small), Sc, 1)

    # both paths at order 40 on the small batch compute the same tube (hull to summation order)
    a, b = variants[f"recompute_order40_S{Sc}"][0](), variants[f"chain_order40_S{Sc}"][0]()
    torch.cuda.synchronize()
    hull_diff = max(float((a[2][:, -1] - b[2]).abs().max()), float((a[3][:, -1] - b[3]).abs().max()))
    for name, (fn, _, _) in variants.items():     # warm-up: module load, first launch of every shape
        fn()
    torch.cuda.synchronize()
    ms = {name: [] for name in variants}
    for _ in range(args.rounds):
        for name, (fn, _, reps) in variants.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            ms[name].append(e0.elapsed_time(e1) / reps)
    os.environ.pop("TZDDPC_ROLLOUT", None)
    med = {k: float(np.median(v)) for k, v in ms.items()}
    rate = {k: variants[k][1] * steps / med[k] * 1e3 for k in ms}
    out = {"card": card(), "scenarios": S, "chain_scenarios": Sc, "steps": steps, "rounds": args.rounds,
           "ms_per_rollout": {k: [round(q, 3) for q in v] for k, v in ms.items()},
           "median_ms": {k: round(v, 3) for k, v in med.items()},
           "spread": {k: round(max(v) / min(v) - 1.0, 4) for k, v in ms.items()},
           "median_scenario_steps_per_s": {k: float(f"{v:.4g}") for k, v in rate.items()},
           "recompute_over_resident": {o: round(med[f"resident_order{o}"] / med[f"recompute_order{o}"], 3) for o in (10, 20, 30)},
           "recompute_order40_full_over_chain_rate": round(rate["recompute_order40"] / rate[f"chain_order40_S{Sc}"], 2),
           "recompute_order40_over_chain_rate_same_batch": round(rate[f"recompute_order40_S{Sc}"] / rate[f"chain_order40_S{Sc}"], 2),
           "order40_last_hull_max_abs_diff_recompute_vs_chain": hull_diff}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
