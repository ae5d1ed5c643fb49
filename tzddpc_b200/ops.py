"""PyTorch custom ops `torch.ops.tzddpc.*`: thin shims from CUDA tensors to the C ABI.

PyTorch is plumbing here (device memory, streams); the arithmetic is in libtzddpc.so.
Every op is registered for CUDA only -- there is deliberately no CPU kernel.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Tuple

import torch
from torch import Tensor

from . import _abi


@dataclass
class SolverOptions:
    """Mirror of TzSolverOpts (include/tzddpc.h); the reference passes **cvxpy_kwargs (tzddpc/tzddpc.py:361)."""
    rho: float = 0.1
    rho_active: float = 100.0
    rho_inactive: float = 0.1
    sigma: float = 1e-6
    alpha: float = 1.6
    eps_abs: float = 1e-6
    eps_rel: float = 1e-6
    max_iter: int = 4000
    check_every: int = 8
    polish: int = 3          # iterations of the active-set polish, 0 = off
    warm_start: int = 0      # 0 cold, 1 reuse (x, y) of the previous call, 2 active-set hint of the previous call
    cert_first: int = 3      # first ADMM iteration at which the active-set KKT certificate is tried, 0 = off
    tube_packed: int = 0     # 1: Ze[1].Z is written as n_nz rows (Program.tube_pattern) instead of the dense n(1+g1) rows
    hot_path: int = 1        # 1: warm_start == 2 on a two-variable program runs fast_step_kernel first (bit-identical results)

    def pack(self) -> List[float]:
        return [self.rho, self.rho_active, self.rho_inactive, self.sigma, self.alpha, self.eps_abs, self.eps_rel,
                float(self.max_iter), float(self.check_every), float(int(self.polish)), float(self.warm_start),
                float(int(self.cert_first)), float(int(self.tube_packed)), float(int(self.hot_path))]


def _opts(o: List[float]) -> _abi.TzSolverOpts:
    s = _abi.TzSolverOpts()
    s.rho, s.rho_active, s.rho_inactive, s.sigma, s.alpha, s.eps_abs, s.eps_rel = o[:7]
    s.max_iter, s.check_every, s.polish, s.warm_start = int(o[7]), int(o[8]), int(o[9]), int(o[10])
    s.cert_first = int(o[11]) if len(o) > 11 else 3
    s.tube_packed = int(o[12]) if len(o) > 12 else 0
    s.hot_path = int(o[13]) if len(o) > 13 else 1
    return s


def _ptr(t: Optional[Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream(t: Tensor):
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _chk(t: Tensor, dtype=torch.float64):
    assert t.is_cuda and t.dtype == dtype and t.is_contiguous(), "expected a contiguous CUDA tensor of " + str(dtype)


def _chk_opt(t: Optional[Tensor], what: str, shape: Tuple[int, ...], dtype=torch.float64):
    """Optional output / scratch tensors are handed to the kernels as raw pointers: the C ABI cannot know their sizes, so a
    wrong dtype, a non-contiguous slice or a wrong shape would corrupt device memory silently."""
    if t is not None:
        _chk(t, dtype)
        assert tuple(t.shape) == shape, f"{what}: expected {shape}, got {tuple(t.shape)}"


def _chk_W(W: Optional[Tensor], n: int) -> int:
    """The noise zonotope W = [c_W, G_W] (n, 1+gW) of reach_step / tube_rollout, or None; returns gW."""
    if W is None:
        return 0
    assert W.dim() == 2 and W.shape[1] >= 1, f"W: expected ({n}, 1+gW), got {tuple(W.shape)}"
    _chk_opt(W, "W", (n, W.shape[1]))
    return W.shape[1] - 1


def _chk_warm(warm: Optional[Tensor], S: int, min_rows: int, used: bool):
    """The warm-start scratch (rows >= min_rows, S): a CUDA float64 tensor whenever given, its shape checked where `used`."""
    if warm is None:
        return
    _chk(warm)
    if used:
        shape = tuple(warm.shape)
        assert len(shape) == 2 and shape[1] == S, f"warm: expected (rows, {S}), got {shape}"
        assert shape[0] >= min_rows, f"warm: needs at least {min_rows} rows, got {shape[0]}"


def _solve(handle: int, is_set: bool, dims: List[int], xbar0: Tensor, e0: Tensor, warm: Optional[Tensor], want_tube: bool,
           opts: List[float]) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """The body of `solve` (a program) and `solve_set` (a program set, `is_set`)."""
    _chk(xbar0), _chk(e0)
    n, nv, nt, nent = dims
    S = xbar0.shape[1]
    dev = xbar0.device
    cost = torch.empty(S, dtype=torch.float64, device=dev)
    v = torch.empty((nv, S), dtype=torch.float64, device=dev)
    traj = torch.empty((nt, S), dtype=torch.float64, device=dev)
    ze1 = torch.empty((nent if want_tube else 0, S), dtype=torch.float64, device=dev)
    status = torch.empty(S, dtype=torch.int32, device=dev)
    iters = torch.empty(S, dtype=torch.int32, device=dev)
    o = _opts(opts)
    d = _abi.program_dims(handle, is_set)
    assert xbar0.shape == (d[0], S) and e0.shape == xbar0.shape, "xbar0, e0: (n, S)"
    assert (nv, nt) == (d[2], d[3]) and (not want_tube or nent == (d[5] if o.tube_packed else d[4])), "dims do not match the program"
    _chk_warm(warm, S, d[6], bool(o.warm_start))
    name = "tz_solve_set" if is_set else "tz_solve"
    with torch.cuda.device(dev):
        rc = getattr(_abi.lib(), name)(C.c_void_p(handle), C.byref(o), S, _ptr(xbar0), _ptr(e0), _ptr(cost), _ptr(v), _ptr(traj),
                                       _ptr(ze1) if want_tube else None, _ptr(status), _ptr(iters), _ptr(warm), _stream(xbar0))
    _abi.check(rc, name)
    return cost, v, traj, ze1, status, iters


def _closed_loop(handle: int, is_set: bool, steps: Optional[int], x: Tensor, xbar: Tensor, e: Tensor, noise: Tensor,
                 x_restart: Optional[Tensor], plant: Tuple[Tensor, ...], status: Tensor, cost: Optional[Tensor], v: Optional[Tensor],
                 traj: Optional[Tensor], ze1: Optional[Tensor], u: Optional[Tensor], hist: Tuple[Optional[Tensor], ...],
                 iters: Optional[Tensor], warm: Optional[Tensor], stats: Optional[Tensor], opts: List[float]) -> None:
    """The body of every closed-loop op.  `handle` is a program, or a program set with `is_set` (tz_closed_loop_*_set).
    `steps` None is one step (tz_closed_loop_step*); otherwise a fused run of `steps` steps (tz_closed_loop_run*), whose noise
    and per-step outputs carry a leading `steps` dimension and `hist` = (x_hist, xbar_hist, e_hist).  `plant` is
    (A_true, B_true), shared by the batch, or (AB_true,), a plant per scenario (tz_closed_loop_*_plants)."""
    _chk(x), _chk(xbar), _chk(e), _chk(noise), _chk(status, torch.int32)
    S = x.shape[1]
    o = _opts(opts)
    n, m, nv, nt, nent, n_nz, warm_rows = _abi.program_dims(handle, is_set)
    if len(plant) == 2:
        _chk(plant[0]), _chk(plant[1])
    else:
        _chk(plant[0])
        assert tuple(plant[0].shape) == (n * (n + m), S), f"AB_true: expected ({n * (n + m)}, {S}), got {tuple(plant[0].shape)}"
    lead, k, per = ((), 1, "") if steps is None else ((steps,), steps, "steps, ")
    assert k >= 1 and x.shape == (n, S) and xbar.shape == x.shape and e.shape == x.shape, "x, xbar, e: (n, S)"
    assert noise.shape == lead + (n, S), f"noise: ({per}n, S)"
    assert status.shape == lead + (S,), f"status: ({per}S)"
    rows = n_nz if o.tube_packed else nent
    outs = [(cost, "cost", (S,)), (v, "v", (nv, S)), (traj, "traj", (nt, S)), (ze1, "ze1", (rows, S)), (u, "u", (m, S))]
    outs += [(h, what, (n, S)) for h, what in zip(hist, ("x_hist", "xbar_hist", "e_hist"))]
    for t, what, shape in outs:
        _chk_opt(t, what, lead + shape)
    _chk_opt(iters, "iters", lead + (S,), torch.int32)
    _chk_opt(x_restart, "x_restart", (n, S))
    if stats is not None:
        _chk(stats)
        assert stats.numel() >= k * _abi.TZ_NSTATS, f"stats: needs {k} x TZ_NSTATS doubles"
    _chk_warm(warm, S, warm_rows, bool(o.warm_start))
    name = ("tz_closed_loop_step" if steps is None else "tz_closed_loop_run") + ("_set" if is_set else "") + \
        ("_plants" if len(plant) == 1 else "")
    with torch.cuda.device(x.device):
        rc = getattr(_abi.lib(), name)(C.c_void_p(handle), C.byref(o), S, *lead, _ptr(x), _ptr(xbar), _ptr(e), _ptr(noise), _ptr(x_restart),
                                       *map(_ptr, plant), _ptr(cost), _ptr(v), _ptr(traj), _ptr(ze1), _ptr(u), *map(_ptr, hist),
                                       _ptr(status), _ptr(iters), _ptr(warm), _ptr(stats), _stream(x))
    _abi.check(rc, name)


# The ops take no default values: torch strips trailing defaulted arguments, which breaks mutated Optional[Tensor] args.
_STEP_MUTATES = ("x", "xbar", "e", "cost", "v", "traj", "ze1", "u", "status", "iters", "warm", "stats")
_RUN_MUTATES = ("x", "xbar", "e", "cost", "v", "traj", "ze1", "u", "x_hist", "xbar_hist", "e_hist", "status", "iters", "warm", "stats")


@torch.library.custom_op("tzddpc::solve", mutates_args=("warm",), device_types="cuda")
def solve(prog: int, dims: List[int], xbar0: Tensor, e0: Tensor, warm: Optional[Tensor], want_tube: bool,
          opts: List[float]) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """Batched TZDDPC.solve (tzddpc/tzddpc.py:357-377).  xbar0, e0: (n, S).  dims = [n, nv, (N+1)n, n(1+g1)].
    Returns cost (S), v (nv, S), xbar (., S), Ze1.Z (n(1+g1), S), status (S), iters (S)."""
    return _solve(prog, False, dims, xbar0, e0, warm, want_tube, opts)


@torch.library.custom_op("tzddpc::closed_loop_step", mutates_args=_STEP_MUTATES, device_types="cuda")
def closed_loop_step(prog: int, x: Tensor, xbar: Tensor, e: Tensor, noise: Tensor, x_restart: Optional[Tensor],
                     A_true: Tensor, B_true: Tensor, status: Tensor, cost: Optional[Tensor], v: Optional[Tensor], traj: Optional[Tensor],
                     ze1: Optional[Tensor], u: Optional[Tensor], iters: Optional[Tensor], warm: Optional[Tensor],
                     stats: Optional[Tensor], opts: List[float]) -> None:
    """One fused closed-loop step, in place on (x, xbar, e) -- examples/2.pulley_sim.py:81-96."""
    _closed_loop(prog, False, None, x, xbar, e, noise, x_restart, (A_true, B_true), status, cost, v, traj, ze1, u, (), iters, warm,
                 stats, opts)


@torch.library.custom_op("tzddpc::closed_loop_run", mutates_args=_RUN_MUTATES, device_types="cuda")
def closed_loop_run(prog: int, steps: int, x: Tensor, xbar: Tensor, e: Tensor, noise: Tensor, x_restart: Optional[Tensor],
                    A_true: Tensor, B_true: Tensor, status: Tensor, cost: Optional[Tensor], v: Optional[Tensor], traj: Optional[Tensor],
                    ze1: Optional[Tensor], u: Optional[Tensor], x_hist: Optional[Tensor], xbar_hist: Optional[Tensor], e_hist: Optional[Tensor],
                    iters: Optional[Tensor], warm: Optional[Tensor], stats: Optional[Tensor], opts: List[float]) -> None:
    """`steps` fused closed-loop steps in ONE launch (tz_closed_loop_run): the loop of examples/2.pulley_sim.py:81-96 for a small
    batch.  noise: (steps, n, S); per-step outputs are step-major: status / iters / cost (steps, S), v (steps, nv, S),
    traj (steps, (N+1)n, S), ze1 (steps, rows, S), u (steps, m, S), x_hist / xbar_hist / e_hist (steps, n, S), stats (steps, TZ_NSTATS)."""
    _closed_loop(prog, False, steps, x, xbar, e, noise, x_restart, (A_true, B_true), status, cost, v, traj, ze1, u,
                 (x_hist, xbar_hist, e_hist), iters, warm, stats, opts)


@torch.library.custom_op("tzddpc::closed_loop_step_plants", mutates_args=_STEP_MUTATES, device_types="cuda")
def closed_loop_step_plants(prog: int, x: Tensor, xbar: Tensor, e: Tensor, noise: Tensor, x_restart: Optional[Tensor],
                            AB_true: Tensor, status: Tensor, cost: Optional[Tensor], v: Optional[Tensor], traj: Optional[Tensor],
                            ze1: Optional[Tensor], u: Optional[Tensor], iters: Optional[Tensor], warm: Optional[Tensor],
                            stats: Optional[Tensor], opts: List[float]) -> None:
    """`closed_loop_step` with a plant per scenario: AB_true (n(n+m), S) in place of A_true, B_true; entry (i, k) of scenario s's
    [A_true B_true] at [i (n+m) + k, s] -- the layout sample_plants returns."""
    _closed_loop(prog, False, None, x, xbar, e, noise, x_restart, (AB_true,), status, cost, v, traj, ze1, u, (), iters, warm, stats,
                 opts)


@torch.library.custom_op("tzddpc::closed_loop_run_plants", mutates_args=_RUN_MUTATES, device_types="cuda")
def closed_loop_run_plants(prog: int, steps: int, x: Tensor, xbar: Tensor, e: Tensor, noise: Tensor, x_restart: Optional[Tensor],
                           AB_true: Tensor, status: Tensor, cost: Optional[Tensor], v: Optional[Tensor], traj: Optional[Tensor],
                           ze1: Optional[Tensor], u: Optional[Tensor], x_hist: Optional[Tensor], xbar_hist: Optional[Tensor],
                           e_hist: Optional[Tensor], iters: Optional[Tensor], warm: Optional[Tensor], stats: Optional[Tensor],
                           opts: List[float]) -> None:
    """`closed_loop_run` with a plant per scenario: AB_true (n(n+m), S) in place of A_true, B_true."""
    _closed_loop(prog, False, steps, x, xbar, e, noise, x_restart, (AB_true,), status, cost, v, traj, ze1, u,
                 (x_hist, xbar_hist, e_hist), iters, warm, stats, opts)


@torch.library.custom_op("tzddpc::solve_set", mutates_args=("warm",), device_types="cuda")
def solve_set(pset: int, dims: List[int], xbar0: Tensor, e0: Tensor, warm: Optional[Tensor], want_tube: bool,
              opts: List[float]) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """`solve` over a program set (data-set axis: scenarios [begin[j], begin[j+1]) use the program of data set j).
    dims = [n, nv, (N+1)n, tube rows]."""
    return _solve(pset, True, dims, xbar0, e0, warm, want_tube, opts)


@torch.library.custom_op("tzddpc::closed_loop_step_set", mutates_args=_STEP_MUTATES, device_types="cuda")
def closed_loop_step_set(pset: int, x: Tensor, xbar: Tensor, e: Tensor, noise: Tensor, x_restart: Optional[Tensor],
                         A_true: Tensor, B_true: Tensor, status: Tensor, cost: Optional[Tensor], v: Optional[Tensor],
                         traj: Optional[Tensor], ze1: Optional[Tensor], u: Optional[Tensor], iters: Optional[Tensor],
                         warm: Optional[Tensor], stats: Optional[Tensor], opts: List[float]) -> None:
    """`closed_loop_step` over a program set: every data set's scenarios are stepped with that data set's program, one launch."""
    _closed_loop(pset, True, None, x, xbar, e, noise, x_restart, (A_true, B_true), status, cost, v, traj, ze1, u, (), iters, warm,
                 stats, opts)


@torch.library.custom_op("tzddpc::closed_loop_step_set_plants", mutates_args=_STEP_MUTATES, device_types="cuda")
def closed_loop_step_set_plants(pset: int, x: Tensor, xbar: Tensor, e: Tensor, noise: Tensor, x_restart: Optional[Tensor],
                                AB_true: Tensor, status: Tensor, cost: Optional[Tensor], v: Optional[Tensor], traj: Optional[Tensor],
                                ze1: Optional[Tensor], u: Optional[Tensor], iters: Optional[Tensor], warm: Optional[Tensor],
                                stats: Optional[Tensor], opts: List[float]) -> None:
    """`closed_loop_step_set` with a plant per scenario: AB_true (n(n+m), S) in place of A_true, B_true."""
    _closed_loop(pset, True, None, x, xbar, e, noise, x_restart, (AB_true,), status, cost, v, traj, ze1, u, (), iters, warm, stats,
                 opts)


@torch.library.custom_op("tzddpc::closed_loop_run_set", mutates_args=_RUN_MUTATES, device_types="cuda")
def closed_loop_run_set(pset: int, steps: int, x: Tensor, xbar: Tensor, e: Tensor, noise: Tensor, x_restart: Optional[Tensor],
                        A_true: Tensor, B_true: Tensor, status: Tensor, cost: Optional[Tensor], v: Optional[Tensor], traj: Optional[Tensor],
                        ze1: Optional[Tensor], u: Optional[Tensor], x_hist: Optional[Tensor], xbar_hist: Optional[Tensor],
                        e_hist: Optional[Tensor], iters: Optional[Tensor], warm: Optional[Tensor], stats: Optional[Tensor],
                        opts: List[float]) -> None:
    """`closed_loop_run` over a program set (tz_closed_loop_run_set): `steps` steps of every data set's scenarios in ONE launch,
    bit-equal to `steps` calls of `closed_loop_step_set`; the layout of `closed_loop_run`."""
    _closed_loop(pset, True, steps, x, xbar, e, noise, x_restart, (A_true, B_true), status, cost, v, traj, ze1, u,
                 (x_hist, xbar_hist, e_hist), iters, warm, stats, opts)


@torch.library.custom_op("tzddpc::closed_loop_run_set_plants", mutates_args=_RUN_MUTATES, device_types="cuda")
def closed_loop_run_set_plants(pset: int, steps: int, x: Tensor, xbar: Tensor, e: Tensor, noise: Tensor, x_restart: Optional[Tensor],
                               AB_true: Tensor, status: Tensor, cost: Optional[Tensor], v: Optional[Tensor], traj: Optional[Tensor],
                               ze1: Optional[Tensor], u: Optional[Tensor], x_hist: Optional[Tensor], xbar_hist: Optional[Tensor],
                               e_hist: Optional[Tensor], iters: Optional[Tensor], warm: Optional[Tensor], stats: Optional[Tensor],
                               opts: List[float]) -> None:
    """`closed_loop_run_set` with a plant per scenario: AB_true (n(n+m), S) in place of A_true, B_true."""
    _closed_loop(pset, True, steps, x, xbar, e, noise, x_restart, (AB_true,), status, cost, v, traj, ze1, u,
                 (x_hist, xbar_hist, e_hist), iters, warm, stats, opts)


@torch.library.custom_op("tzddpc::interval_hull", mutates_args=(), device_types="cuda")
def interval_hull(Z: Tensor) -> Tuple[Tensor, Tensor]:
    """Z: (S, n, 1+g) -> lo, hi (S, n).  Zonotope.interval (tzddpc/tzddpc.py:191-197)."""
    _chk(Z)
    S, n, ld = Z.shape
    lo = torch.empty((S, n), dtype=torch.float64, device=Z.device)
    hi = torch.empty_like(lo)
    with torch.cuda.device(Z.device):
        rc = _abi.lib().tz_interval_hull(S, n, ld - 1, _ptr(Z), _ptr(lo), _ptr(hi), _stream(Z))
    _abi.check(rc, "tz_interval_hull")
    return lo, hi


@torch.library.custom_op("tzddpc::reach_step", mutates_args=(), device_types="cuda")
def reach_step(Cm: Tensor, Gm: Tensor, Z: Tensor, W: Optional[Tensor]) -> Tensor:
    """MatrixZonotope x Zonotope (+ W).  Cm: (n, p) or (S, n, p); Gm: (N, n, p) or (S, N, n, p);
    Z: (S, p, 1+g); W: (n, 1+gW).  Returns (S, n, (N+1)(1+g)+gW)  (tzddpc/tzddpc.py:175-176,181,185,205).
    Every shape is checked here: the C ABI takes raw pointers, and a per-scenario Cm needs a per-scenario Gm."""
    _chk(Z)
    assert Z.dim() == 3, f"Z: expected (S, p, 1+g), got {tuple(Z.shape)}"
    S, p, ld = Z.shape
    per = Cm.dim() == 3
    lead = (S,) if per else ()
    assert Cm.dim() in (2, 3) and Cm.shape[-2] >= 1, f"Cm: expected (n, {p}) or ({S}, n, {p}), got {tuple(Cm.shape)}"
    n = Cm.shape[-2]
    _chk_opt(Cm, "Cm", lead + (n, p))
    assert Gm.dim() == len(lead) + 3, f"Gm: expected {lead + ('N', n, p)} (shared / per scenario as Cm), got {tuple(Gm.shape)}"
    N = Gm.shape[-3]
    _chk_opt(Gm, "Gm", lead + (N, n, p))
    gW = _chk_W(W, n)
    out = torch.empty((S, n, (N + 1) * ld + gW), dtype=torch.float64, device=Z.device)
    with torch.cuda.device(Z.device):
        rc = _abi.lib().tz_reach_step(S, n, p, N, ld - 1, gW, _ptr(Cm), _ptr(Gm), int(per), _ptr(Z), _ptr(W), _ptr(out),
                                      _stream(Z))
    _abi.check(rc, "tz_reach_step")
    return out


@torch.library.custom_op("tzddpc::girard_reduce", mutates_args=(), device_types="cuda")
def girard_reduce(Z: Tensor, order: float, metric: int, gout_cap: int) -> Tuple[Tensor, Tensor]:
    """Z: (S, n, 1+g) -> (S, n, 1+gout_cap), gout (S).  Zonotope.reduce (SURVEY App. A.5)."""
    _chk(Z)
    S, n, ld = Z.shape
    out = torch.empty((S, n, 1 + gout_cap), dtype=torch.float64, device=Z.device)
    gout = torch.empty(S, dtype=torch.int32, device=Z.device)
    with torch.cuda.device(Z.device):
        rc = _abi.lib().tz_girard_reduce(S, n, ld - 1, float(order), int(metric), _ptr(Z), gout_cap, _ptr(out), _ptr(gout),
                                         _stream(Z))
    _abi.check(rc, "tz_girard_reduce")
    return out, gout


@torch.library.custom_op("tzddpc::tube_rollout", mutates_args=(), device_types="cuda")
def tube_rollout(CK: Tensor, GK: Tensor, GD: Tensor, Z0: Tensor, XU: Tensor, W: Optional[Tensor], order: float, metric: int,
                 gcap: int) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """Z_{k+1} = reduce(M_K x Z_k + M_Delta x <[xbar_k; v_k], 0> + W, order) for k < steps, zonotope resident in shared
    memory (tzddpc/tzddpc.py:175-186,205 + Zonotope.reduce).  CK: (n, n) or (S, n, n); GK: (NK, n, n) or (S, NK, n, n);
    GD: (ND, n, n+m) or (S, ND, n, n+m); Z0: (S, n, 1+g0); XU: (S, steps, n+m); W: (n, 1+gW).
    Returns Zfinal (S, n, 1+gcap), gfinal (S), hull_lo, hull_hi (S, steps, n).
    Where the pre-reduction generator block fits in shared memory (order <= 31 for the 5-dim stress system) it is built
    there every step (tube_rollout_kernel); beyond that its entries are recomputed wherever the Girard reduction reads them
    (tube_rollout_recompute_kernel, order <= 135 there), with the same results bit for bit.  Larger orders raise, naming the
    bytes both kernels need.  TZDDPC_ROLLOUT=resident / recompute forces one kernel where it fits (include/tzddpc.h).
    Every shape is checked here, as in reach_step: a per-scenario CK needs per-scenario GK and GD."""
    _chk(Z0), _chk(XU)
    assert Z0.dim() == 3 and Z0.shape[1] >= 1, f"Z0: expected (S, n, 1+g0), got {tuple(Z0.shape)}"
    S, n, ld0 = Z0.shape
    assert XU.dim() == 3 and XU.shape[0] == S and XU.shape[2] > n, f"XU: expected ({S}, steps, {n}+m), got {tuple(XU.shape)}"
    steps, p = XU.shape[1], XU.shape[2]
    per = CK.dim() == 3
    lead = (S,) if per else ()
    _chk_opt(CK, "CK", lead + (n, n))
    assert GK.dim() == len(lead) + 3, f"GK: expected {lead + ('NK', n, n)} (shared / per scenario as CK), got {tuple(GK.shape)}"
    assert GD.dim() == len(lead) + 3, f"GD: expected {lead + ('ND', n, p)} (shared / per scenario as CK), got {tuple(GD.shape)}"
    NK, ND = GK.shape[-3], GD.shape[-3]
    _chk_opt(GK, "GK", lead + (NK, n, n))
    _chk_opt(GD, "GD", lead + (ND, n, p))
    gW = _chk_W(W, n)
    dev = Z0.device
    Zf = torch.empty((S, n, 1 + gcap), dtype=torch.float64, device=dev)
    gf = torch.empty(S, dtype=torch.int32, device=dev)
    lo = torch.empty((S, steps, n), dtype=torch.float64, device=dev)
    hi = torch.empty_like(lo)
    with torch.cuda.device(dev):
        rc = _abi.lib().tz_tube_rollout(S, n, p - n, NK, ND, gW, ld0 - 1, steps, float(order), int(metric), _ptr(CK), _ptr(GK),
                                        _ptr(GD), int(per), _ptr(Z0), _ptr(XU), _ptr(W), int(gcap), _ptr(Zf), _ptr(gf),
                                        _ptr(lo), _ptr(hi), _stream(Z0))
    _abi.check(rc, "tz_tube_rollout")
    return Zf, gf, lo, hi


@torch.library.custom_op("tzddpc::sample_noise", mutates_args=(), device_types="cuda")
def sample_noise(WZ: Tensor, S: int, vertex: bool, seed: int, scenario_offset: int, t: int) -> Tensor:
    """Closed-loop noise of step t for S scenarios: (n, S) = c_W + G_W beta, Philox stream keyed by `seed`, counter
    (scenario_offset + s, t).  W.sample() (examples/2.pulley_sim.py:92) or a random vertex (examples/1.double_integrator_sim.py:85)."""
    _chk(WZ)
    n = WZ.shape[0]
    out = torch.empty((n, S), dtype=torch.float64, device=WZ.device)
    with torch.cuda.device(WZ.device):
        rc = _abi.lib().tz_sample_noise(S, S, n, WZ.shape[1] - 1, _ptr(WZ), int(vertex), seed, scenario_offset, t, _ptr(out), _stream(WZ))
    _abi.check(rc, "tz_sample_noise")
    return out


@torch.library.custom_op("tzddpc::generate_trajectories", mutates_args=(), device_types="cuda")
def generate_trajectories(A: Tensor, B: Tensor, X0Z: Tensor, UZ: Tensor, WZ: Tensor, S: int, T: int, seed: int,
                          scenario_offset: int) -> Tuple[Tensor, Tensor]:
    """examples/utils.py:6-45 batched over S data sets on the device.  A (n, n), B (n, m) shared by the data sets, or
    A (S, n, n), B (S, n, m): data set s from the plant (A[s], B[s]).  Returns U (S, T, m), X (S, T, n)."""
    _chk(A), _chk(B), _chk(X0Z), _chk(UZ), _chk(WZ)
    per = B.dim() == 3
    n, m = B.shape[-2:]
    if per:
        assert tuple(A.shape) == (S, n, n) and B.shape[0] == S, f"A, B: expected ({S}, n, n), ({S}, n, m), got {tuple(A.shape)}, {tuple(B.shape)}"
    else:
        assert tuple(A.shape) == (n, n) and B.dim() == 2, f"A, B: expected (n, n), (n, m), got {tuple(A.shape)}, {tuple(B.shape)}"
    assert X0Z.shape[0] == n and WZ.shape[0] == n and UZ.shape[0] == m, "X0Z, WZ: n rows, UZ: m rows"
    U = torch.empty((S, T, m), dtype=torch.float64, device=A.device)
    X = torch.empty((S, T, n), dtype=torch.float64, device=A.device)
    fn = _abi.lib().tz_generate_trajectories_plants if per else _abi.lib().tz_generate_trajectories
    with torch.cuda.device(A.device):
        rc = fn(S, T, n, m, X0Z.shape[1] - 1, UZ.shape[1] - 1, WZ.shape[1] - 1, _ptr(A), _ptr(B),
                _ptr(X0Z), _ptr(UZ), _ptr(WZ), seed, scenario_offset, _ptr(U), _ptr(X), _stream(A))
    _abi.check(rc, "tz_generate_trajectories_plants" if per else "tz_generate_trajectories")
    return U, X


@torch.library.custom_op("tzddpc::sample_plants", mutates_args=(), device_types="cuda")
def sample_plants(AB: Tensor, Pinv: Tensor, WZ: Tensor, dataset: Optional[Tensor], S: int, seed: int, scenario_offset: int) -> Tensor:
    """S plants drawn from the un-reduced model sets M_Sigma = (X1 - M_w) pinv([X0; U0]) of D data sets (tz_sample_plants):
    AB (D, n, n+m), Pinv (D, T-1, n+m) as `identify` returns them, WZ (n, 1+gW); dataset (S,) int32 -- the data set of every
    scenario -- or None (data set 0).  Philox stream (seed, scenario_offset + s, purpose 6).  Returns AB_true (n(n+m), S), the
    layout of the *_plants closed-loop ops."""
    _chk(AB), _chk(Pinv), _chk(WZ)
    D, n, nm = AB.shape
    assert Pinv.dim() == 3 and Pinv.shape[0] == D and Pinv.shape[2] == nm, f"Pinv: expected ({D}, T-1, {nm}), got {tuple(Pinv.shape)}"
    assert WZ.dim() == 2 and WZ.shape[0] == n, f"WZ: expected ({n}, 1+gW), got {tuple(WZ.shape)}"
    if dataset is not None:
        _chk(dataset, torch.int32)
        assert tuple(dataset.shape) == (S,), f"dataset: expected ({S},), got {tuple(dataset.shape)}"
    out = torch.empty((n * nm, S), dtype=torch.float64, device=AB.device)
    with torch.cuda.device(AB.device):
        rc = _abi.lib().tz_sample_plants(S, D, Pinv.shape[1] + 1, n, nm - n, WZ.shape[1] - 1, _ptr(AB), _ptr(Pinv), _ptr(WZ),
                                         _ptr(dataset), int(seed), int(scenario_offset), _ptr(out), _stream(AB))
    _abi.check(rc, "tz_sample_plants")
    return out


@torch.library.custom_op("tzddpc::identify", mutates_args=(), device_types="cuda")
def identify(X: Tensor, U: Tensor, WZ: Tensor, K: Optional[Tensor], want_pinv: bool) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """X: (S, T, n), U: (S, T, m), WZ: (n, 1+gW), K: (S, m, n).  Returns AB (S,n,n+m), dAB, dK (S,n,n), Pinv, status.
    M_Sigma = (X1 - M_w) pinv([X0;U0]) and its order-1 boxes (tzddpc/tzddpc.py:81-83,119-128)."""
    _chk(X), _chk(U), _chk(WZ)
    S, T, n = X.shape
    m = U.shape[2]
    dev = X.device
    AB = torch.empty((S, n, n + m), dtype=torch.float64, device=dev)
    dAB = torch.empty_like(AB)
    dK = torch.zeros((S, n, n), dtype=torch.float64, device=dev)
    Pinv = torch.empty((S, T - 1, n + m) if want_pinv else (0,), dtype=torch.float64, device=dev)
    status = torch.empty(S, dtype=torch.int32, device=dev)
    if K is not None:
        _chk(K)
    with torch.cuda.device(dev):
        rc = _abi.lib().tz_identify(S, T, n, m, WZ.shape[1] - 1, _ptr(X), _ptr(U), _ptr(WZ), _ptr(K), _ptr(AB), _ptr(dAB),
                                    _ptr(dK) if K is not None else None, _ptr(Pinv) if want_pinv else None,
                                    _ptr(status), _stream(X))
    _abi.check(rc, "tz_identify")
    return AB, dAB, dK, Pinv, status


@torch.library.custom_op("tzddpc::gain_synthesis", mutates_args=(), device_types="cuda")
def gain_synthesis(AB: Tensor, Pinv: Tensor, WZ: Tensor, tol: float, max_iter: int, num_init: int, accuracy: float,
                   confidence: float, seed: int, dataset_offset: int) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """compute_theta + is_gain_robust (tzddpc/utils.py:58-129) batched over D data sets.  AB: (D, n, n+m), Pinv: (D, T-1, n+m),
    WZ: (n, 1+gW).  Returns K (D, m, n), dA (D, n, n), dB (D, n, m), rho (D, 3), robust, iters, status (D, int32)."""
    _chk(AB), _chk(Pinv), _chk(WZ)
    D, n, d = AB.shape
    m, Tm = d - n, Pinv.shape[1]
    dev = AB.device
    f64 = dict(dtype=torch.float64, device=dev)
    K, dA, dB, rho = torch.empty((D, m, n), **f64), torch.empty((D, n, n), **f64), torch.empty((D, n, m), **f64), torch.empty((D, 3), **f64)
    robust, iters, status = (torch.empty(D, dtype=torch.int32, device=dev) for _ in range(3))
    with torch.cuda.device(dev):
        rc = _abi.lib().tz_gain_synthesis(D, Tm + 1, n, m, WZ.shape[1] - 1, _ptr(AB), _ptr(Pinv), _ptr(WZ), float(tol), int(max_iter),
                                          int(num_init), float(accuracy), float(confidence), int(seed), int(dataset_offset),
                                          _ptr(K), _ptr(dA), _ptr(dB), _ptr(rho), _ptr(robust), _ptr(iters), _ptr(status), _stream(AB))
    _abi.check(rc, "tz_gain_synthesis")
    return K, dA, dB, rho, robust, iters, status


@torch.library.custom_op("tzddpc::gain_adversary", mutates_args=(), device_types="cuda")
def gain_adversary(AB: Tensor, Pinv: Tensor, WZ: Tensor, K: Tensor, num_init: int, accuracy: float, confidence: float,
                   seed: int, dataset_offset: int) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """compute_A_B + is_gain_robust (tzddpc/utils.py:13-41,105-129) for given gains K (D, m, n), batched over D data sets.
    Returns dA (D, n, n), dB (D, n, m), rho (D, 3), robust, status (D, int32)."""
    _chk(AB), _chk(Pinv), _chk(WZ), _chk(K)
    D, n, d = AB.shape
    m, Tm = d - n, Pinv.shape[1]
    dev = AB.device
    f64 = dict(dtype=torch.float64, device=dev)
    dA, dB, rho = torch.empty((D, n, n), **f64), torch.empty((D, n, m), **f64), torch.empty((D, 3), **f64)
    robust, status = (torch.empty(D, dtype=torch.int32, device=dev) for _ in range(2))
    with torch.cuda.device(dev):
        rc = _abi.lib().tz_gain_adversary(D, Tm + 1, n, m, WZ.shape[1] - 1, _ptr(AB), _ptr(Pinv), _ptr(WZ), _ptr(K), int(num_init),
                                          float(accuracy), float(confidence), int(seed), int(dataset_offset),
                                          _ptr(dA), _ptr(dB), _ptr(rho), _ptr(robust), _ptr(status), _stream(AB))
    _abi.check(rc, "tz_gain_adversary")
    return dA, dB, rho, robust, status


@torch.library.custom_op("tzddpc::qp_solve", mutates_args=(), device_types="cuda")
def qp_solve(prog: int, q: Tensor, l: Tensor, u: Tensor, opts: List[float]) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """Explicit-instance batched ADMM: q (nz, S), l/u (nc, S) -> z (nz, S), y (nc, S), status, iters."""
    _chk(q), _chk(l), _chk(u)
    S = q.shape[1]
    z = torch.empty_like(q)
    y = torch.empty_like(l)
    status = torch.empty(S, dtype=torch.int32, device=q.device)
    iters = torch.empty(S, dtype=torch.int32, device=q.device)
    o = _opts(opts)
    with torch.cuda.device(q.device):
        rc = _abi.lib().tz_qp_solve(C.c_void_p(prog), C.byref(o), S, _ptr(q), _ptr(l), _ptr(u), _ptr(z), _ptr(y),
                                    _ptr(status), _ptr(iters), _stream(q))
    _abi.check(rc, "tz_qp_solve")
    return z, y, status, iters
