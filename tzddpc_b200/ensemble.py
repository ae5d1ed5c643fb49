"""`TZDDPCEnsemble` -- the data-set axis of the scenario batch (BASELINE.json north_star: scenarios = noise realisations
x initial states x data sets).

The reference builds one `TZDDPC` object per data set -- one model M_Sigma (`tzddpc/tzddpc.py:67-85`), one gain, one
problem (`:132-241`) -- and runs the closed loops one after another (`examples/2.pulley_sim.py:62-103` repeats the whole
script per run).  Here D controllers of identical structure are fused into a *program set* (`tz_program_set_create`):
scenarios `[begin[j], begin[j+1])` of the batch are stepped with the program of data set j, all in ONE kernel launch per
closed-loop step (`tz_closed_loop_step_set`), or -- below `FUSED_RUN_MAX_BATCH` scenarios -- in one launch for the whole
run (`tz_closed_loop_run_set`).
"""
from __future__ import annotations

from typing import Optional, Sequence, Union

import numpy as np
import torch

from . import _abi, ops
from .objects import Data, SystemZonotopes
from .ops import SolverOptions
from .tzddpc import TZDDPC


class _SetProgram:
    """Duck-typed stand-in for `_abi.Program` (handle / warm_rows / compiled / tube_pattern / bucket) backed by a program set."""

    def __init__(self, pset: _abi.ProgramSet):
        p0 = pset.programs[0]
        self.pset = pset
        self.handle = pset.handle
        self.warm_rows, self.compiled, self.tube_pattern, self.bucket = p0.warm_rows, p0.compiled, p0.tube_pattern, p0.bucket


def _canonicalise_chunks(canon, D: int, chunk: int = 256):
    """compile_program_batch over [0, D) in chunks of `chunk` data sets on a thread pool (numpy releases the GIL in its
    element-wise loops); the chunks must agree on the structure, and are concatenated along the data-set axis."""
    import dataclasses
    from concurrent.futures import ThreadPoolExecutor
    import os
    bounds = [(lo, min(lo + chunk, D)) for lo in range(0, D, chunk)]
    if len(bounds) == 1:
        return canon(0, D)
    with ThreadPoolExecutor(max_workers=min(len(bounds), max(1, len(os.sched_getaffinity(0))))) as ex:
        parts = list(ex.map(lambda b: canon(*b), bounds))
    p0 = parts[0]
    fields = {}
    for f in dataclasses.fields(p0):
        v0 = getattr(p0, f.name)
        if isinstance(v0, np.ndarray) and f.name not in ("ze1_ptr", "ze1_idx"):
            for q in parts[1:]:
                assert getattr(q, f.name).shape[1:] == v0.shape[1:], f"data sets differ in structure ({f.name})"
            fields[f.name] = np.concatenate([getattr(q, f.name) for q in parts], axis=0)
        else:
            for q in parts[1:]:
                same = np.array_equal(getattr(q, f.name), v0) if isinstance(v0, np.ndarray) else getattr(q, f.name) == v0
                assert same, f"data sets differ in structure ({f.name})"
            fields[f.name] = v0
    return type(p0)(**fields)


def _abi_batch(cbatch, K, device):
    with torch.cuda.device(device):
        return _abi.ProgramBatch(cbatch, K)


class _DeviceData:
    """D data sets living on the device as U (D, T, m), X (D, T, n); item d is fetched to the host on demand."""

    def __init__(self, U, X):
        self.U, self.X = U, X

    def __len__(self):
        return self.X.shape[0]

    def __getitem__(self, d):
        return Data(self.U[d].cpu().numpy(), self.X[d].cpu().numpy())


class _LazyControllers:
    """`ensemble.controllers` of an ensemble built in one go: controller d (a TZDDPC that owns nothing on the device, its
    program is a view into the ensemble's batch) is materialised on first access."""

    def __init__(self, ens, datasets, zonotopes, AB, dAB, dK, thetas, horizon):
        self._ens, self._data, self._z, self._AB, self._dAB, self._dK, self._th, self._h = ens, datasets, zonotopes, AB, dAB, dK, thetas, horizon
        self._made = {}

    def __len__(self):
        return len(self._data)

    def __getitem__(self, d):
        d = int(d)
        if d < 0:
            d += len(self)
        if d not in self._made:
            c = TZDDPC(self._data[d], device=self._ens.device)
            c.verbose = False
            ok = c._adopt_model(self._z, self._AB[d], self._dAB[d], self._dK[d], self._th[d])
            assert ok
            c._Pinv = None if self._ens._Pinv is None else self._ens._Pinv[d]
            c._program = self._ens._batch.programs[d]
            c.problem_full, c.horizon = c._program, self._h
            c.parameters, c.variables = ("e0", "xbar0"), ("v", "xbar", "Ze")
            c._dims = list(self._ens._dims)
            self._made[d] = c
        return self._made[d]

    def __iter__(self):
        return (self[d] for d in range(len(self)))


class TZDDPCEnsemble(object):
    _solve_op = staticmethod(ops.solve_set)
    _step_ops = (ops.closed_loop_step_set, ops.closed_loop_step_set_plants)
    _run_ops = (ops.closed_loop_run_set, ops.closed_loop_run_set_plants)
    # below FUSED_RUN_MAX_BATCH scenarios `simulate` runs the whole loop in one launch (tz_closed_loop_run_set), as TZDDPC does
    FUSED_RUN_MAX_BATCH = TZDDPC.FUSED_RUN_MAX_BATCH
    _fused_run_ok = TZDDPC._fused_run_ok

    def __init__(self, controllers: Sequence[TZDDPC], scenarios_per_dataset: Union[int, Sequence[int]]):
        """controllers: D `TZDDPC` objects on which `build_problem` has been called with the same horizon, cost and
        constraints (one per data set).  scenarios_per_dataset: scenarios of each data set (an int, or one count per data
        set; every count but the last must be a multiple of 16)."""
        assert len(controllers) >= 1
        c0 = controllers[0]
        for c in controllers:
            assert c._program is not None, "call build_problem on every controller first"
            assert (c.dim_x, c.dim_u, c.horizon, c.device) == (c0.dim_x, c0.dim_u, c0.horizon, c0.device)
        D = len(controllers)
        counts = [int(scenarios_per_dataset)] * D if np.isscalar(scenarios_per_dataset) else [int(v) for v in scenarios_per_dataset]
        assert len(counts) == D and all(v >= 0 for v in counts)
        assert all(v % 16 == 0 for v in counts[:-1]), "scenarios per data set must be a multiple of 16 (all but the last)"
        self.controllers = list(controllers)
        self.begin = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
        with torch.cuda.device(c0.device):                # the set's entry table lives on the controllers' device
            self._program = _SetProgram(_abi.ProgramSet([c._program for c in controllers], self.begin))
        self.device, self.solver_options, self.verbose = c0.device, SolverOptions(), False
        self.dim_x, self.dim_u, self.horizon, self._dims = c0.dim_x, c0.dim_u, c0.horizon, list(c0._dims)
        self.zonotopes = c0.zonotopes
        self.num_scenarios = int(self.begin[-1])
        # the data sets' models for sample_plants (controllers whose model was adopted from elsewhere carry no pseudo-inverse)
        pinvs = [getattr(c, "_Pinv", None) for c in controllers]
        ok = all(p_ is not None and p_.shape == pinvs[0].shape for p_ in pinvs)
        self._ABd = c0._t(np.stack([c._AB for c in controllers])) if ok else None
        self._Pinv = torch.stack(pinvs).contiguous() if ok else None

    @classmethod
    def from_datasets(cls, datasets: Sequence[Data], zonotopes: SystemZonotopes, horizon: int, build_loss, build_constraints=None,
                      scenarios_per_dataset: Union[int, Sequence[int]] = 16, K: Optional[np.ndarray] = None, k0: Optional[int] = None,
                      device=None, tol: float = 1e-5, num_max_iterations: int = 20, num_initial_points: int = 10,
                      accuracy: float = 1e-2, confidence: float = 1e-5, seed: int = 25) -> "TZDDPCEnsemble":
        """What the reference does once per data set -- TZDDPC(data), build_zonotopes_theta, build_problem
        (examples/2.pulley_sim.py:59-75) -- for D data sets of equal length, with the device work batched over the data sets:
        ONE tz_identify launch (model + pseudo-inverse), ONE tz_gain_synthesis launch (a gain per data set; or `K`, (m, n)
        shared / (D, m, n) per data set), ONE tz_identify launch for the boxes of M_K; then the host canonicalisation batched
        over the data sets and ONE tz_program_create_batch.
        `datasets`: a sequence of Data, or a pair of CUDA tensors (U (D, T, m), X (D, T, n)) -- e.g. straight from
        ops.generate_trajectories -- which never leave the device."""
        import torch
        if isinstance(datasets, tuple) and len(datasets) == 2 and isinstance(datasets[0], torch.Tensor):
            U, X = datasets[0].contiguous(), datasets[1].contiguous()
            datasets = _DeviceData(U, X)
            c0 = TZDDPC(datasets[0], device=X.device)
        else:
            datasets = list(datasets)
            c0 = TZDDPC(datasets[0], device=device)
            for d_ in datasets:
                assert np.asarray(d_.x).shape == np.asarray(datasets[0].x).shape and np.asarray(d_.u).shape == np.asarray(datasets[0].u).shape, \
                    "data sets must have the same shape"
            X = c0._t(np.stack([np.asarray(d_.x, dtype=np.float64) for d_ in datasets]))        # (one upload for all data sets)
            U = c0._t(np.stack([np.asarray(d_.u, dtype=np.float64) for d_ in datasets]))
        c0.verbose = False
        D, n, m = len(datasets), c0.dim_x, c0.dim_u
        WZ = c0._t(zonotopes.W.Z)
        AB, dAB, _, Pinv, status = ops.identify(X, U, WZ, None, True)
        if int((status != 0).sum().item()) != 0:
            raise Exception('Identification failed: [X0; U0] does not have full row rank')
        info = None
        if K is None:
            Kd, dA, dB, rho, robust, iters, st = ops.gain_synthesis(AB, Pinv, WZ, tol, num_max_iterations, num_initial_points,
                                                                    accuracy, confidence, seed, 0)
            if int((st != 0).sum().item()) != 0:
                raise Exception('Gain synthesis failed: a Riccati iteration did not converge')
            assert bool(robust.bool().all().item()), f'K is not robust with accuracy-confidence of {accuracy, 1 - confidence}'
            info = {"rho": rho.cpu().numpy(), "iterations": iters.cpu().numpy(), "robust": robust.cpu().numpy().astype(bool)}
            dA_h, dB_h = dA.cpu().numpy(), dB.cpu().numpy()
        else:
            Kh = np.asarray(K, dtype=np.float64)
            Kd = c0._t(np.broadcast_to(Kh.reshape((-1, m, n)) if Kh.ndim == 3 else Kh.reshape(1, m, n), (D, m, n)))
            dA_h, dB_h = np.zeros((D, n, n)), np.zeros((D, n, m))
        _, _, dK, _, _ = ops.identify(X, U, WZ, Kd.contiguous(), False)
        AB_h, dAB_h, dK_h, K_h = AB.cpu().numpy(), dAB.cpu().numpy(), dK.cpu().numpy(), Kd.cpu().numpy()
        from .objects import Theta
        thetas = [Theta(K_h[d].copy(), dA_h[d], dB_h[d]) for d in range(D)]
        boxed = zonotopes.W.num_generators * (c0.num_samples - 1) > n * (n + m)
        if not boxed:
            # data sets so short that reduce(1) is a no-op (SURVEY.md App. A.5): the dense generators, one controller at a time
            ctls = [TZDDPC(datasets[d], device=c0.device) for d in range(D)]
            for d, c in enumerate(ctls):
                c.verbose = False
                c.build_zonotopes_theta(zonotopes, K=K_h[d])
                c._build(int(horizon), build_loss, build_constraints, k0)
            ens = cls(ctls, scenarios_per_dataset)
            ens.theta_info = info
            return ens
        # ---- the D programs in one go: batched host canonicalisation (program.compile_program_batch: the structural
        # decisions once, the arithmetic vectorised over the data sets, chunks on a thread pool), then ONE
        # tz_program_create_batch (packed on the host, one upload).  Controllers are materialised on demand.
        from .program import TubeModelBatch, compile_program_batch
        cost, box = c0._resolve(build_loss, build_constraints, int(horizon), k0 is not None)
        Xi, Ui = zonotopes.X.interval, zonotopes.U.interval
        WZh = np.asarray(zonotopes.W.Z, dtype=np.float64)

        def canon(lo, hi):
            mb = TubeModelBatch.boxed(AB_h[lo:hi], dAB_h[lo:hi], dK_h[lo:hi], K_h[lo:hi], WZh, Xi.left_limit, Xi.right_limit,
                                      Ui.left_limit, Ui.right_limit)
            return compile_program_batch(mb, int(horizon), cost, box, k0=k0)

        cbatch = _canonicalise_chunks(canon, D)
        pbatch = _abi_batch(cbatch, K_h, c0.device)
        ens = cls.__new__(cls)
        ens._ABd, ens._Pinv = AB, Pinv
        ens._init_from_batch(pbatch, datasets, zonotopes, AB_h, dAB_h, dK_h, thetas, int(horizon), scenarios_per_dataset, c0.device)
        ens.theta_info = info
        return ens

    def _init_from_batch(self, pbatch, datasets, zonotopes, AB, dAB, dK, thetas, horizon, scenarios_per_dataset, device):
        D = pbatch.num
        counts = [int(scenarios_per_dataset)] * D if np.isscalar(scenarios_per_dataset) else [int(v) for v in scenarios_per_dataset]
        assert len(counts) == D and all(v >= 0 for v in counts)
        assert all(v % 16 == 0 for v in counts[:-1]), "scenarios per data set must be a multiple of 16 (all but the last)"
        self._batch = pbatch
        self.begin = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
        with torch.cuda.device(device):
            self._program = _SetProgram(_abi.ProgramSet(pbatch.programs, self.begin))
        self.device, self.solver_options, self.verbose = device, SolverOptions(), False
        cb = pbatch.compiled
        self.dim_x, self.dim_u, self.horizon = cb.n, cb.m, horizon
        self._dims = [cb.n, cb.nv, (horizon + 1) * cb.n, cb.n * (1 + cb.g1)]
        self.zonotopes = zonotopes
        self.num_scenarios = int(self.begin[-1])
        self._K = np.stack([t.K for t in thetas])
        self.controllers = _LazyControllers(self, datasets, zonotopes, AB, dAB, dK, thetas, horizon)

    @property
    def num_datasets(self) -> int:
        return len(self.begin) - 1

    def dataset_of(self) -> np.ndarray:
        """data set index of every scenario of the batch"""
        return np.repeat(np.arange(self.num_datasets), np.diff(self.begin))

    @property
    def K(self) -> np.ndarray:
        """(D, m, n) feedback gains theta.K of the data sets"""
        if getattr(self, "_K", None) is not None:
            return self._K
        return np.stack([c.theta.K for c in self.controllers])

    _t = TZDDPC._t
    solve_batch = TZDDPC.solve_batch
    _plant_batch = TZDDPC._plant_batch
    _split_plants = TZDDPC._split_plants

    def sample_plants(self, seed: int, scenario_offset: int = 0):
        """A plant per scenario, drawn from the model set M_Sigma of the scenario's own data set (as TZDDPC.sample_plants; the
        draws of scenario s are those of global scenario scenario_offset + s).  Returns CUDA tensors A (S, n, n), B (S, n, m)."""
        if getattr(self, "_Pinv", None) is None:
            raise RuntimeError("sample_plants needs every data set's pseudo-inverse pinv([X0; U0]); these controllers carry none "
                               "(build them with build_zonotopes, or the ensemble with from_datasets)")
        S = self.num_scenarios
        ds = torch.as_tensor(self.dataset_of().astype(np.int32), device=self.device)
        AB = ops.sample_plants(self._ABd, self._Pinv, self._t(self.zonotopes.W.Z), ds, S, int(seed), int(scenario_offset))
        return self._split_plants(AB)

    def simulate(self, A_true, B_true, x0, *args, **kwargs):
        x0 = np.atleast_2d(np.asarray(x0, dtype=np.float64))
        assert x0.shape[0] == self.num_scenarios, f"x0 must have one row per scenario ({self.num_scenarios})"
        return TZDDPC.simulate(self, A_true, B_true, x0, *args, **kwargs)

    simulate.__doc__ = TZDDPC.simulate.__doc__
