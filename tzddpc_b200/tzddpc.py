"""`TZDDPC` -- drop-in counterpart of the reference controller class (`tzddpc/tzddpc.py:11-500`).

Same public methods, properties and attributes; behind them every numeric step runs on the
GPU (sm_100a) through `torch.ops.tzddpc.*` -> libtzddpc.so:

  build_zonotopes / build_zonotopes_theta  -> tz_identify            (tzddpc/tzddpc.py:67-130)
  build_problem / build_problem_simplified -> host canonicalisation (program.py) + tz_program_create
                                                                     (tzddpc/tzddpc.py:132-355)
  solve                                    -> tz_solve               (tzddpc/tzddpc.py:357-377)
  simulate (new, batched closed loop)      -> tz_closed_loop_step    (examples/2.pulley_sim.py:81-96)

Additive extensions: `solve` accepts (S, n) batches; `simulate` runs S scenarios in lock step.
Deviations (documented in DESIGN.md): the loss/constraint callbacks receive this package's
affine-expression variables (`tzddpc_b200.cvx`) instead of cvxpy ones, or a structured
`StageCost`/`BoxConstraint`; `compute_theta` needs K from the caller or uses an LQR gain
(the reference's SDP + DCCP/MOSEK synthesis, tzddpc/utils.py:13-103, is out of scope).
"""
from __future__ import annotations

from typing import Callable, List, Optional, Tuple, Union

import numpy as np
import torch

from . import _abi, ops
from .objects import Data, DataDrivenDataset, OptimizationProblem, SystemZonotopes, Theta
from .ops import SolverOptions
from .program import BoxConstraint, CompiledProgram, StageCost, TubeModel, compile_program
from .zonotope import Interval, MatrixZonotope, Zonotope, boxed_generators, concatenate_zonotope


class _Value:
    """Mimics a cvxpy expression's `.value` (callers read `Ze[1].Z.value`, examples/2.pulley_sim.py:96)."""

    def __init__(self, value):
        self.value = value


class TubeHandle:
    """What `solve` returns in place of the reference's `CVXZonotope` Ze[1] (`tzddpc/tzddpc.py:377`):
    `.Z.value` is the n x (1+g1) array [c, G] (batched: S x n x (1+g1)), fetched from the GPU lazily -- as the
    reference's `.Z.value` evaluates its expression on access (examples/2.pulley_sim.py:96).
    With `pattern` the device buffer is the packed tube (`SolverOptions.tube_packed`): row i = entry pattern[i] of Ze[1].Z,
    every other entry is structurally zero; `.Z.value` scatters it into the dense matrix on the host."""

    def __init__(self, ze1: torch.Tensor, n: int, g1: int, batched: bool, pattern: Optional[np.ndarray] = None):
        self._ze1, self._n, self._g1, self._batched, self._pattern = ze1, n, g1, batched, pattern
        self._host = None

    @property
    def Z(self) -> _Value:
        if self._host is None:
            S = self._ze1.shape[1]
            if self._pattern is None:
                a = self._ze1.reshape(self._n, 1 + self._g1, S).permute(2, 0, 1).cpu().numpy()
            else:
                a = np.zeros((S, self._n * (1 + self._g1)))
                a[:, self._pattern] = self._ze1.t().cpu().numpy()
                a = a.reshape(S, self._n, 1 + self._g1)
            self._host = a if self._batched else a[0]
        return _Value(self._host)

    @property
    def device_tensor(self) -> torch.Tensor:
        """(n, 1+g1, S) view of the device buffer (entry (r, j) of scenario s at [r, j, s]); packed tubes are expanded."""
        if self._pattern is not None:
            S = self._ze1.shape[1]
            d = torch.zeros((self._n * (1 + self._g1), S), dtype=torch.float64, device=self._ze1.device)
            d[torch.as_tensor(self._pattern, dtype=torch.long, device=d.device)] = self._ze1
            return d.reshape(self._n, 1 + self._g1, -1)
        return self._ze1.reshape(self._n, 1 + self._g1, -1)

    @property
    def center(self) -> _Value:
        return _Value(self.Z.value[..., 0])

    @property
    def generators(self) -> _Value:
        return _Value(self.Z.value[..., 1:])

    @property
    def num_generators(self) -> int:
        return self._g1


class BatchSolveResult:
    def __init__(self, cost, v, xbar, tube, status, iters):
        self.cost, self.v, self.xbar, self.tube, self.status, self.iters = cost, v, xbar, tube, status, iters


class TZDDPC(object):
    optimization_problem: Union[OptimizationProblem, None] = None
    dataset: DataDrivenDataset
    zonotopes: SystemZonotopes
    Mdata: MatrixZonotope
    Mdelta: MatrixZonotope
    MdataK: MatrixZonotope
    theta: Theta

    # the launch entry points (TZDDPCEnsemble swaps in the program-set variants); the step ops and the fused-run ops, each for
    # a shared plant and for a plant per scenario
    _solve_op = staticmethod(ops.solve)
    _step_ops = (ops.closed_loop_step, ops.closed_loop_step_plants)
    _run_ops = (ops.closed_loop_run, ops.closed_loop_run_plants)

    def __init__(self, data: Data, device: Optional[Union[str, torch.device]] = None):
        """:param data: input/state data, each T x dim (tzddpc/tzddpc.py:20-28)."""
        _abi.lib()                               # fail loudly when the CUDA library is missing
        if not torch.cuda.is_available():
            raise RuntimeError("tzddpc_b200.TZDDPC needs a CUDA device (no CPU fallback)")
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.solver_options = SolverOptions()
        self.verbose = True
        self._program: Optional[_abi.Program] = None
        self.update_identification_data(data)

    # ---- tzddpc/tzddpc.py:30-43 -------------------------------------------------------------
    @property
    def num_samples(self) -> int:
        return self.dataset.Um.shape[0] + 1

    @property
    def dim_u(self) -> int:
        return self.dataset.Um.shape[1]

    @property
    def dim_x(self) -> int:
        return self.dataset.Xp.shape[1]

    # ---- tzddpc/tzddpc.py:45-65 -------------------------------------------------------------
    def update_identification_data(self, data: Data):
        assert len(data.u.shape) == 2, \
            "Data needs to be shaped as a TxM matrix (T is the number of samples and M is the number of features)"
        assert len(data.x.shape) == 2, \
            "Data needs to be shaped as a TxM matrix (T is the number of samples and M is the number of features)"
        assert data.x.shape[0] == data.u.shape[0], "Input/state data must have the same length"
        Xm, Xp, Um = data.x[:-1], data.x[1:], data.u[:-1]
        self.dataset = DataDrivenDataset(Xp, Xm, Um, data)
        self.optimization_problem = None
        self._program = None

    def _t(self, a) -> torch.Tensor:
        return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).to(self.device)

    # ---- tzddpc/tzddpc.py:67-85 -------------------------------------------------------------
    def build_zonotopes(self, zonotopes: SystemZonotopes) -> MatrixZonotope:
        X0, W, U, X = zonotopes.X0, zonotopes.W, zonotopes.U, zonotopes.X
        assert X0.dimension == W.dimension and X0.dimension == self.dim_x \
            and X.dimension == X0.dimension, 'The zonotopes do not have the correct dimension'
        if self.verbose:
            print('--------------------------------------------')
            print('Building zonotopes')
        self.optimization_problem = None
        self._program = None
        self.zonotopes = zonotopes
        d = self.dataset.original_data
        AB, dAB, _, Pinv, status = ops.identify(self._t(d.x)[None], self._t(d.u)[None], self._t(W.Z), None, True)
        if int(status[0].item()) != 0:
            raise Exception('Identification failed: [X0; U0] does not have full row rank')
        self._AB = AB[0].cpu().numpy()
        self._dAB = dAB[0].cpu().numpy()
        self._Pinv = Pinv[0]                                   # (T-1) x (n+m), stays on the GPU
        # generators -g_i P[j,:] (rank one; generator index outer, sample index inner -- App. A.7)
        GW = self._t(W.generators)                              # n x gW
        gens = -(GW.t()[:, None, :, None] * self._Pinv[None, :, None, :])       # gW x (T-1) x n x (n+m)
        self.Mdata = MatrixZonotope(self._AB, gens.reshape(-1, self.dim_x, self.dim_x + self.dim_u).cpu().numpy())
        self.Mdata.rank_one = (self._Pinv, self._t(W.Z))       # structure the utils.* gain helpers work on (utils.py)
        if self.verbose:
            print('--------------------------------------------')
        return self.Mdata

    # ---- tzddpc/tzddpc.py:87-93 -------------------------------------------------------------
    def compute_theta(self, tol: float = 1e-5, num_max_iterations: int = 20, num_initial_points: int = 10,
                      K: Optional[np.ndarray] = None, accuracy: float = 1e-2, confidence: float = 1e-5, seed: int = 25) -> Theta:
        """tzddpc/tzddpc.py:87-93 -> tzddpc/utils.py:58-103.  The reference alternates an LMI feasibility SDP with a
        DCCP/MOSEK adversary; that stack is absent and its gain is solver-dependent.  With `K` the caller's gain is used as
        is (Theta's deltas are zero).  Without it the batched GPU synthesis `tz_gain_synthesis` runs the same alternation
        (LQR gain of the adversarial pair, closed-form convex-concave adversary, Monte-Carlo robustness check) and fills
        Theta(K, An - A0, Bn - B0); the reference's assertion `K is not robust` (utils.py:100) is kept."""
        assert self.Mdata is not None, 'Mdata is not defined'
        n, m = self.dim_x, self.dim_u
        if K is not None:
            self.theta = Theta(np.asarray(K, dtype=np.float64).reshape(m, n), np.zeros((n, n)), np.zeros((n, m)))
            return self.theta
        Kd, dA, dB, rho, robust, iters, status = ops.gain_synthesis(
            self._t(self._AB)[None], self._Pinv[None].contiguous(), self._t(self.zonotopes.W.Z), tol, num_max_iterations,
            num_initial_points, accuracy, confidence, seed, 0)
        if int(status[0].item()) != 0:
            raise Exception('Gain synthesis failed: the Riccati iteration of the identified pair did not converge')
        self.theta_info = {"rho_center": float(rho[0, 0]), "rho_adversarial": float(rho[0, 1]), "rho_sampled_max": float(rho[0, 2]),
                           "iterations": int(iters[0]), "robust": bool(robust[0].item())}
        if self.verbose:
            print(f'Optimization completed. Closed loop spectral radius: {max(self.theta_info["rho_center"], self.theta_info["rho_adversarial"])}'
                  f' - K {Kd[0].flatten().tolist()}')
        assert self.theta_info["robust"], f'K is not robust with accuracy-confidence of {accuracy, 1 - confidence}'
        self.theta = Theta(Kd[0].cpu().numpy(), dA[0].cpu().numpy(), dB[0].cpu().numpy())
        return self.theta

    # ---- tzddpc/tzddpc.py:95-130 ------------------------------------------------------------
    def build_zonotopes_theta(self, zonotopes: SystemZonotopes, tol: float = 1e-5, num_max_iterations: int = 20,
                              num_initial_points: int = 10, K: Optional[np.ndarray] = None
                              ) -> Tuple[Theta, MatrixZonotope]:
        self.build_zonotopes(zonotopes)
        self.compute_theta(tol, num_max_iterations, num_initial_points, K=K)
        n, m = self.dim_x, self.dim_u
        d = self.dataset.original_data
        W = zonotopes.W
        num_raw = W.num_generators * (self.num_samples - 1)
        if num_raw > n * (n + m):
            # order-1 Girard reduction boxes every generator; closed form on the GPU (SURVEY App. A.6)
            AB, dAB, dK, _, status = ops.identify(self._t(d.x)[None], self._t(d.u)[None], self._t(W.Z),
                                                  self._t(self.theta.K)[None], False)
            dAB_h, dK_h = dAB[0].cpu().numpy(), dK[0].cpu().numpy()
            centreK = MatrixZonotope(self._AB, np.zeros((0, n, n + m))) * np.vstack([np.eye(n), self.theta.K])
            self.MdataK = MatrixZonotope(centreK.center, boxed_generators(dK_h))                   # :119,127
            self.Mdelta = MatrixZonotope(np.zeros((n, n + m)), boxed_generators(dAB_h))            # :122-123,128
            self.Mdata = MatrixZonotope(self._AB, boxed_generators(dAB_h))                         # :126
        else:
            # tiny data sets: reduce(1) is a no-op (App. A.5), keep the dense generators
            MK = self.Mdata * np.vstack([np.eye(n), self.theta.K])
            Mdelta = self.Mdata + (-1.0 * self._AB)
            self.Mdata, self.MdataK, self.Mdelta = self.Mdata.reduce(1), MK.reduce(1), Mdelta.reduce(1)
        return self.theta, self.Mdata

    def _adopt_model(self, zonotopes: SystemZonotopes, AB: np.ndarray, dAB: np.ndarray, dK: np.ndarray, theta: Theta) -> bool:
        """Takes an identified model computed elsewhere (TZDDPCEnsemble.from_datasets: one batched launch for all data sets)
        in place of build_zonotopes_theta.  Only for the boxed branch (order-1 reduction boxes every generator); returns False
        when the data set is so short that reduce(1) is a no-op and the caller must use build_zonotopes_theta."""
        n, m = self.dim_x, self.dim_u
        if zonotopes.W.num_generators * (self.num_samples - 1) <= n * (n + m):
            return False
        self.optimization_problem, self._program = None, None
        self.zonotopes, self.theta = zonotopes, theta
        self._AB, self._dAB, self._Pinv = AB, dAB, None
        centreK = MatrixZonotope(AB, np.zeros((0, n, n + m))) * np.vstack([np.eye(n), theta.K])
        self.MdataK = MatrixZonotope(centreK.center, boxed_generators(dK))                      # tzddpc/tzddpc.py:119,127
        self.Mdelta = MatrixZonotope(np.zeros((n, n + m)), boxed_generators(dAB))               # :122-123,128
        self.Mdata = MatrixZonotope(AB, boxed_generators(dAB))                                  # :126
        return True

    # ---- tzddpc/tzddpc.py:132-241 / 243-355 -------------------------------------------------
    def _model(self) -> TubeModel:
        X, U = self.zonotopes.X.interval, self.zonotopes.U.interval
        return TubeModel(AB=self.Mdata.center, Acl=self.MdataK.center, GK=self.MdataK.generators,
                         GD=self.Mdelta.generators, K=self.theta.K, WZ=self.zonotopes.W.Z,
                         X_lo=X.left_limit, X_hi=X.right_limit, U_lo=U.left_limit, U_hi=U.right_limit)

    def _resolve(self, build_loss, build_constraints, horizon: int, simplified: bool):
        from . import cvx
        n, m = self.dim_x, self.dim_u
        if isinstance(build_loss, StageCost):
            cost = build_loss
        else:
            assert build_loss is not None, "Loss function callback cannot be none"
            cost = cvx.extract_stage_cost(build_loss, horizon, n, m, simplified)
        if isinstance(build_constraints, BoxConstraint):
            box = build_constraints
        else:
            # quirk Q1: the reference iterates the fallback `(None, None)` and raises (tzddpc/tzddpc.py:213-217)
            if build_constraints is None:
                raise Exception('Constraint 0 is not defined or is not convex.')
            box = cvx.extract_box_constraints(build_constraints, horizon, n, m, simplified)
        return cost, box

    def _build(self, horizon: int, build_loss, build_constraints, k0: Optional[int]):
        cost, box = self._resolve(build_loss, build_constraints, horizon, k0 is not None)
        prog = compile_program(self._model(), horizon, cost, box, k0=k0)
        if self.verbose:
            for k, g in enumerate(prog.gens_per_step):           # tzddpc/tzddpc.py:190,206
                print(f'Step {k}')
                print(g)
        with torch.cuda.device(self.device):             # the program image lives on the controller's device
            self._program = _abi.Program(prog, self.theta.K)
        self.problem_full = self._program
        self.horizon = horizon
        self.parameters = ("e0", "xbar0")
        self.variables = ("v", "xbar", "Ze")
        self._dims = [self.dim_x, prog.nv, (horizon + 1) * self.dim_x, self.dim_x * (1 + prog.g1)]
        return self.problem_full

    def build_problem(self, horizon: int, build_loss, build_constraints=None, **kwargs):
        return self._build(int(horizon), build_loss, build_constraints, None)

    def build_problem_simplified(self, k0: int, horizon: int, build_loss, build_constraints=None, **kwargs):
        return self._build(int(horizon), build_loss, build_constraints, int(k0))

    # ---- tzddpc/tzddpc.py:357-377 -----------------------------------------------------------
    def solve_batch(self, xbar0: torch.Tensor, e0: torch.Tensor, want_tube: bool = True,
                    warm: Optional[torch.Tensor] = None, options: Optional[SolverOptions] = None) -> BatchSolveResult:
        """xbar0, e0: (n, S) float64 CUDA tensors (scenario-fastest)."""
        assert self._program is not None, "call build_problem first"
        o = options or self.solver_options
        pattern = self._program.tube_pattern if o.tube_packed else None
        dims = self._dims[:3] + [len(pattern) if o.tube_packed else self._dims[3]]
        cost, v, traj, ze1, status, iters = self._solve_op(self._program.handle.value, dims, xbar0, e0, warm,
                                                           want_tube, o.pack())
        tube = TubeHandle(ze1, self.dim_x, self._program.compiled.g1, True, pattern) if want_tube else None
        return BatchSolveResult(cost, v, traj, tube, status, iters)

    def solve(self, xbar0: np.ndarray, e0: np.ndarray, **kwargs):
        """Batch 1 (1-D inputs): the reference's return tuple `(result, v, xbar, Ze[1])`.
        Batched ((S, n) inputs): `(cost[S], v[S,N,m], xbar[S,N+1,n], tube, status[S])`."""
        n, m, N = self.dim_x, self.dim_u, self.horizon
        xb = np.asarray(xbar0, dtype=np.float64)
        ee = np.asarray(e0, dtype=np.float64)
        batched = xb.ndim == 2
        xb2, ee2 = np.atleast_2d(xb), np.atleast_2d(ee)
        assert xb2.shape[1] == n and ee2.shape == xb2.shape, "Invalid size"
        r = self.solve_batch(self._t(xb2.T), self._t(ee2.T))
        status = r.status.cpu().numpy()
        cost = r.cost.cpu().numpy()
        v = r.v.cpu().numpy().T.reshape(-1, N, m)
        xbar = r.xbar.cpu().numpy().T.reshape(-1, N + 1, n)
        if batched:
            return cost, v, xbar, r.tube, status
        if status[0] == _abi.TZ_STATUS_NONFINITE:
            with open('zpc_logs.txt', 'w') as f:                             # tzddpc/tzddpc.py:368-371
                print('Error while solving the TZDDPC problem. Details: non-finite data', file=f)
            raise Exception('Error while solving the TZDDPC problem. Details: non-finite data')
        if status[0] == _abi.TZ_STATUS_MAXITER:
            # the reference surfaces a solver failure as an exception (cp.SolverError -> tzddpc/tzddpc.py:366-371)
            with open('zpc_logs.txt', 'w') as f:
                print('Error while solving the TZDDPC problem. Details: the solver did not converge', file=f)
            raise Exception('Error while solving the TZDDPC problem. Details: the solver did not converge')
        if np.isinf(cost[0]):
            raise Exception('Problem is unbounded')                          # tzddpc/tzddpc.py:374-375
        tube = TubeHandle(r.tube._ze1, n, self._program.compiled.g1, False, r.tube._pattern)
        return float(cost[0]), v[0], xbar[0], tube

    # ---- batched closed loop (examples/2.pulley_sim.py:62-103, one scenario per column) --------
    #: batches below this many scenarios run `simulate` as one fused launch (csrc/tz_fused.cu: kHotMinBatch -- from there on
    #: the two-kernel hot path is faster than the step loop inside step_kernel)
    FUSED_RUN_MAX_BATCH = 256

    def _fused_run_ok(self, S: int, steps: int) -> bool:
        return steps >= 2 and S < self.FUSED_RUN_MAX_BATCH and str(self._program.bucket)[:2] in ("B0", "B1", "B2", "B3")

    def _plant_batch(self, A_true, B_true, S: int):
        """The simulated plant as the closed-loop ops take it: (A, B) for one plant (n, n), (n, m) shared by the batch;
        (AB_true,) for a plant per scenario, A_true (S, n, n) and B_true (S, n, m) as numpy arrays or CUDA tensors, with
        AB_true the (n(n+m), S) array of the *_plants ops."""
        ndim = lambda a: a.dim() if isinstance(a, torch.Tensor) else np.ndim(a)          # noqa: E731
        if ndim(A_true) == 2 and ndim(B_true) == 2:
            return self._t(A_true), self._t(B_true)
        n, m = self.dim_x, self.dim_u
        dev = lambda a: a.to(self.device, torch.float64) if isinstance(a, torch.Tensor) else self._t(a)     # noqa: E731
        A, B = dev(A_true), dev(B_true)
        assert tuple(A.shape) == (S, n, n) and tuple(B.shape) == (S, n, m), \
            f"A_true, B_true: expected (n, n), (n, m) or ({S}, {n}, {n}), ({S}, {n}, {m}); got {tuple(A.shape)}, {tuple(B.shape)}"
        return (torch.cat([A, B], dim=2).reshape(S, n * (n + m)).t().contiguous(),)

    def _split_plants(self, AB_true: torch.Tensor):
        """(n(n+m), S) -> A (S, n, n), B (S, n, m)"""
        n, m = self.dim_x, self.dim_u
        AB = AB_true.t().reshape(-1, n, n + m)
        return AB[:, :, :n].contiguous(), AB[:, :, n:].contiguous()

    def sample_plants(self, S: int, seed: int, scenario_offset: int = 0):
        """S plants [A B] drawn uniformly from the generator box of the data-consistent model set
        M_Sigma = (X1 - M_w) pinv([X0; U0]) (tzddpc/tzddpc.py:81-83; the un-reduced set, whose every member the tube covers),
        from the Philox stream (seed, scenario_offset + scenario, purpose 6): a scenario's plant does not depend on how the
        batch is split.  Returns CUDA tensors A (S, n, n), B (S, n, m), for `simulate`."""
        if getattr(self, "_Pinv", None) is None:
            raise RuntimeError("sample_plants needs the pseudo-inverse pinv([X0; U0]) of the data: call build_zonotopes first")
        AB = ops.sample_plants(self._t(self._AB)[None], self._Pinv[None].contiguous(), self._t(self.zonotopes.W.Z), None, int(S),
                               int(seed), int(scenario_offset))
        return self._split_plants(AB)

    def simulate(self, A_true: np.ndarray, B_true: np.ndarray, x0: np.ndarray, noise=None, keep_tubes: bool = False,
                 options: Optional[SolverOptions] = None, restart: bool = False, steps: Optional[int] = None,
                 seed: Optional[int] = None, vertex_noise: bool = False, scenario_offset: int = 0):
        """Run the closed loop for S scenarios in lock step.
        A_true (n, n), B_true (n, m): the plant of every scenario; or A_true (S, n, n), B_true (S, n, m) (numpy arrays or CUDA
        tensors, e.g. from `sample_plants`): scenario s runs on (A_true[s], B_true[s]).
        x0: (S, n); noise: (steps, S, n) array or CUDA tensor (steps, n, S) -- or None with `steps` and `seed`: the noise
        w_t = W.sample() (examples/2.pulley_sim.py:92; a random vertex of W with vertex_noise, examples/1.double_integrator_sim.py:85)
        is then drawn on the device from the Philox stream (seed, scenario_offset + scenario, t), so that a scenario sees the
        same realisation however the batch is sharded over GPUs.
        restart: an infeasible scenario (the reference raises and the run ends, tzddpc/tzddpc.py:374-375) starts a
        new run from its x0 instead of keeping its state.
        Returns dict with x (steps+1, S, n), xbar, e, u, v0, cost (steps, S), status (steps, S), stats (steps, 8)."""
        assert self._program is not None, "call build_problem first"
        n, m = self.dim_x, self.dim_u
        o = options or self.solver_options
        x0 = np.atleast_2d(np.asarray(x0, dtype=np.float64))
        S = x0.shape[0]
        if noise is None:
            assert steps is not None and seed is not None, "give either `noise` or `steps` and `seed`"
            WZ = self._t(self.zonotopes.W.Z)
            w = torch.stack([ops.sample_noise(WZ, S, bool(vertex_noise), int(seed), int(scenario_offset), t) for t in range(steps)])
        elif isinstance(noise, torch.Tensor):
            w = noise
        else:
            w = self._t(np.transpose(np.asarray(noise, dtype=np.float64), (0, 2, 1)))
        steps = w.shape[0]
        dev = self.device
        f64 = dict(dtype=torch.float64, device=dev)
        x, xbar = self._t(x0.T), self._t(x0.T)
        e = torch.zeros((n, S), **f64)
        plant = self._plant_batch(A_true, B_true, S)
        per_scenario = len(plant) == 1
        xs = torch.empty((steps + 1, n, S), **f64)
        xbars = torch.empty_like(xs)
        es = torch.empty_like(xs)
        us = torch.empty((steps, m, S), **f64)
        vs = torch.empty((steps, self._dims[1], S), **f64)
        costs = torch.empty((steps, S), **f64)
        stat = torch.empty((steps, S), dtype=torch.int32, device=dev)
        iters = torch.empty((steps, S), dtype=torch.int32, device=dev)
        stats = torch.zeros((steps, _abi.TZ_NSTATS), **f64)
        pattern = self._program.tube_pattern if o.tube_packed else None
        tubes = torch.empty((steps, len(pattern) if o.tube_packed else self._dims[3], S), **f64) if keep_tubes else None
        warm = torch.zeros((self._program.warm_rows, S), **f64) if o.warm_start else None
        xs[0], xbars[0], es[0] = x, xbar, e
        xr = x.clone() if restart else None
        h = self._program.handle.value
        if self._fused_run_ok(S, steps):
            # small batch: the whole run in ONE launch (tz_closed_loop_run / _run_set; bit-equal to the step loop below)
            run = self._run_ops[per_scenario]
            run(h, steps, x, xbar, e, w.contiguous(), xr, *plant, stat, costs, vs, None, tubes, us, xs[1:], xbars[1:], es[1:], iters, warm,
                stats, o.pack())
        else:
            step = self._step_ops[per_scenario]
            for t in range(steps):
                step(h, x, xbar, e, w[t].contiguous(), xr, *plant, stat[t], costs[t], vs[t], None, tubes[t] if keep_tubes else None, us[t],
                     iters[t], warm, stats[t], o.pack())
                xs[t + 1], xbars[t + 1], es[t + 1] = x, xbar, e
        out = {"x": xs.permute(0, 2, 1).cpu().numpy(), "xbar": xbars.permute(0, 2, 1).cpu().numpy(),
               "e": es.permute(0, 2, 1).cpu().numpy(), "u": us.permute(0, 2, 1).cpu().numpy(),
               "v": vs.permute(0, 2, 1).cpu().numpy(), "cost": costs.cpu().numpy(), "status": stat.cpu().numpy(),
               "iters": iters.cpu().numpy(), "stats": stats.cpu().numpy()}
        if keep_tubes:
            g1 = self._program.compiled.g1
            if pattern is None:
                out["tubes"] = tubes.reshape(steps, n, 1 + g1, S).permute(0, 3, 1, 2).cpu().numpy()
            else:
                dense = np.zeros((steps, S, n * (1 + g1)))
                dense[:, :, pattern] = tubes.permute(0, 2, 1).cpu().numpy()
                out["tubes"] = dense.reshape(steps, S, n, 1 + g1)
        return out
