"""ctypes binding of libtzddpc.so (include/tzddpc.h).  No fallback: if the library is
missing the import of the hot path fails loudly."""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

import os

LIB_PATH = Path(os.environ.get("TZDDPC_LIB", Path(__file__).resolve().parent / "lib" / "libtzddpc.so"))

TZ_OK = 0
TZ_STATUS_OK, TZ_STATUS_MAXITER, TZ_STATUS_INFEASIBLE, TZ_STATUS_NONFINITE = 0, 1, 2, 3
TZ_NSTATS = 8

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)


class TzProgramDesc(C.Structure):
    _fields_ = [(k, C.c_int32) for k in ("n", "m", "horizon", "nv", "nz", "nc", "npar", "na", "nchk", "nkink", "g1", "nterms")] + \
               [(k, C.c_void_p) for k in ("P", "q0", "Qp", "A", "l0", "u0", "kink0", "wabs", "R", "Bt", "gam", "Rchk", "cc",
                                          "CC2", "XB", "ze1_ptr", "ze1_idx", "ze1_val", "D", "E")] + \
               [("c", C.c_double), ("K", C.c_void_p)]


class TzSolverOpts(C.Structure):
    _fields_ = [(k, C.c_double) for k in ("rho", "rho_active", "rho_inactive", "sigma", "alpha", "eps_abs", "eps_rel")] + \
               [(k, C.c_int32) for k in ("max_iter", "check_every", "polish", "warm_start", "cert_first", "tube_packed", "hot_path")]


class TzddpcLibraryMissing(RuntimeError):
    pass


_lib = None

# every symbol include/tzddpc.h declares (tests/test_abi.py checks the library exports all of them)
EXPORTS = ["tz_version", "tz_last_error", "tz_device_cc", "tz_program_create", "tz_program_destroy", "tz_program_bucket", "tz_program_warm_rows",
           "tz_solver_opts_default", "tz_solve", "tz_closed_loop_step", "tz_closed_loop_step_host_scratch_bytes",
           "tz_closed_loop_step_host", "tz_interval_hull", "tz_reach_step", "tz_girard_reduce", "tz_tube_rollout",
           "tz_identify", "tz_qp_solve", "tz_philox4x32_10_host", "tz_sample_noise", "tz_generate_trajectories",
           "tz_program_tube_pattern", "tz_program_set_create", "tz_program_set_destroy", "tz_program_set_scenarios",
           "tz_solve_set", "tz_closed_loop_step_set", "tz_gain_synthesis", "tz_gain_robust_samples", "tz_gain_adversary", "tz_program_dims",
           "tz_program_set_dims", "tz_closed_loop_run_host", "tz_program_create_batch",
           "tz_program_batch_get", "tz_program_batch_destroy", "tz_closed_loop_run", "tz_closed_loop_step_plants",
           "tz_closed_loop_step_set_plants", "tz_closed_loop_run_plants", "tz_sample_plants", "tz_generate_trajectories_plants",
           "tz_closed_loop_run_set", "tz_closed_loop_run_set_plants"]


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise TzddpcLibraryMissing(
            f"{LIB_PATH} not found: the TZDDPC hot path has no CPU fallback. Build it with "
            f"`python -m tzddpc_b200.build` (needs nvcc; cross-compiles for sm_100a without a GPU).")
    L = C.CDLL(str(LIB_PATH))
    vp, i64, i32, dbl = C.c_void_p, C.c_int64, C.c_int32, C.c_double
    L.tz_version.restype = C.c_char_p
    L.tz_last_error.restype = C.c_size_t
    L.tz_last_error.argtypes = [C.c_char_p, C.c_size_t]
    L.tz_device_cc.restype = C.c_int
    L.tz_program_create.restype = C.c_int
    L.tz_program_create.argtypes = [C.POINTER(TzProgramDesc), C.POINTER(vp)]
    L.tz_program_create_batch.restype = C.c_int
    L.tz_program_create_batch.argtypes = [C.POINTER(TzProgramDesc), i32, C.POINTER(vp)]
    L.tz_program_batch_get.restype = vp
    L.tz_program_batch_get.argtypes = [vp, i32]
    L.tz_program_batch_destroy.restype = None
    L.tz_program_batch_destroy.argtypes = [vp]
    L.tz_program_destroy.restype = None
    L.tz_program_destroy.argtypes = [vp]
    L.tz_program_bucket.restype = C.c_int
    L.tz_program_bucket.argtypes = [vp, C.c_char_p, C.c_size_t]
    L.tz_program_warm_rows.restype = C.c_int
    L.tz_program_warm_rows.argtypes = [vp]
    L.tz_solver_opts_default.restype = None
    L.tz_solver_opts_default.argtypes = [C.POINTER(TzSolverOpts)]
    L.tz_solve.restype = C.c_int
    L.tz_solve.argtypes = [vp, C.POINTER(TzSolverOpts), i64] + [vp] * 10
    L.tz_closed_loop_step.restype = C.c_int
    L.tz_closed_loop_step.argtypes = [vp, C.POINTER(TzSolverOpts), i64] + [vp] * 17
    L.tz_closed_loop_run.restype = C.c_int
    L.tz_closed_loop_run.argtypes = [vp, C.POINTER(TzSolverOpts), i64, C.c_int32] + [vp] * 20
    L.tz_closed_loop_step_plants.restype = C.c_int
    L.tz_closed_loop_step_plants.argtypes = [vp, C.POINTER(TzSolverOpts), i64] + [vp] * 16
    L.tz_closed_loop_run_plants.restype = C.c_int
    L.tz_closed_loop_run_plants.argtypes = [vp, C.POINTER(TzSolverOpts), i64, C.c_int32] + [vp] * 19
    L.tz_program_dims.restype = C.c_int
    L.tz_program_dims.argtypes = [vp, vp]
    L.tz_program_set_dims.restype = C.c_int
    L.tz_program_set_dims.argtypes = [vp, vp]
    L.tz_program_tube_pattern.restype = C.c_int
    L.tz_program_tube_pattern.argtypes = [vp, vp, i32]
    L.tz_program_set_create.restype = C.c_int
    L.tz_program_set_create.argtypes = [vp, i32, vp, C.POINTER(vp)]
    L.tz_program_set_destroy.restype = None
    L.tz_program_set_destroy.argtypes = [vp]
    L.tz_program_set_scenarios.restype = i64
    L.tz_program_set_scenarios.argtypes = [vp]
    L.tz_solve_set.restype = C.c_int
    L.tz_solve_set.argtypes = [vp, C.POINTER(TzSolverOpts), i64] + [vp] * 10
    L.tz_closed_loop_step_set.restype = C.c_int
    L.tz_closed_loop_step_set.argtypes = [vp, C.POINTER(TzSolverOpts), i64] + [vp] * 17
    L.tz_closed_loop_step_set_plants.restype = C.c_int
    L.tz_closed_loop_step_set_plants.argtypes = [vp, C.POINTER(TzSolverOpts), i64] + [vp] * 16
    L.tz_closed_loop_run_set.restype = C.c_int
    L.tz_closed_loop_run_set.argtypes = [vp, C.POINTER(TzSolverOpts), i64, C.c_int32] + [vp] * 20
    L.tz_closed_loop_run_set_plants.restype = C.c_int
    L.tz_closed_loop_run_set_plants.argtypes = [vp, C.POINTER(TzSolverOpts), i64, C.c_int32] + [vp] * 19
    L.tz_closed_loop_step_host_scratch_bytes.restype = C.c_size_t
    L.tz_closed_loop_step_host_scratch_bytes.argtypes = [vp, i64]
    L.tz_closed_loop_step_host.restype = C.c_int
    L.tz_closed_loop_step_host.argtypes = [vp, C.POINTER(TzSolverOpts), i64] + [vp] * 12 + [i32]
    L.tz_closed_loop_run_host.restype = C.c_int
    L.tz_closed_loop_run_host.argtypes = [vp, C.POINTER(TzSolverOpts), i64, i32] + [vp] * 14 + [i32]
    L.tz_interval_hull.restype = C.c_int
    L.tz_interval_hull.argtypes = [i64, i32, i32, vp, vp, vp, vp]
    L.tz_reach_step.restype = C.c_int
    L.tz_reach_step.argtypes = [i64, i32, i32, i32, i32, i32, vp, vp, i32, vp, vp, vp, vp]
    L.tz_girard_reduce.restype = C.c_int
    L.tz_girard_reduce.argtypes = [i64, i32, i32, dbl, i32, vp, i32, vp, vp, vp]
    L.tz_tube_rollout.restype = C.c_int
    L.tz_tube_rollout.argtypes = [i64] + [i32] * 7 + [dbl, i32, vp, vp, vp, i32, vp, vp, vp, i32, vp, vp, vp, vp, vp]
    u32, u64 = C.c_uint32, C.c_uint64
    L.tz_philox4x32_10_host.restype = None
    L.tz_philox4x32_10_host.argtypes = [u32] * 6 + [C.POINTER(u32)]
    L.tz_sample_noise.restype = C.c_int
    L.tz_sample_noise.argtypes = [i64, i64, i32, i32, vp, i32, u64, i64, u32, vp, vp]
    L.tz_generate_trajectories.restype = C.c_int
    L.tz_generate_trajectories.argtypes = [i64] + [i32] * 6 + [vp] * 5 + [u64, i64, vp, vp, vp]
    L.tz_generate_trajectories_plants.restype = C.c_int
    L.tz_generate_trajectories_plants.argtypes = [i64] + [i32] * 6 + [vp] * 5 + [u64, i64, vp, vp, vp]
    L.tz_sample_plants.restype = C.c_int
    L.tz_sample_plants.argtypes = [i64] + [i32] * 5 + [vp] * 4 + [u64, i64, vp, vp]
    L.tz_identify.restype = C.c_int
    L.tz_identify.argtypes = [i64, i32, i32, i32, i32] + [vp] * 10
    L.tz_gain_synthesis.restype = C.c_int
    L.tz_gain_synthesis.argtypes = [i64, i32, i32, i32, i32, vp, vp, vp, dbl, i32, i32, dbl, dbl, u64, i64] + [vp] * 8
    L.tz_gain_adversary.restype = C.c_int
    L.tz_gain_adversary.argtypes = [i64, i32, i32, i32, i32, vp, vp, vp, vp, i32, dbl, dbl, u64, i64] + [vp] * 6
    L.tz_gain_robust_samples.restype = i32
    L.tz_gain_robust_samples.argtypes = [dbl, dbl]
    L.tz_qp_solve.restype = C.c_int
    L.tz_qp_solve.argtypes = [vp, C.POINTER(TzSolverOpts), i64] + [vp] * 8
    _lib = L
    return L


def program_dims(handle: int, is_set: bool = False):
    """(n, m, nv, (N+1)n, n(1+g1), n_nz, warm_rows) of a program / program set handle."""
    out = (C.c_int32 * 8)()
    L = lib()
    check((L.tz_program_set_dims if is_set else L.tz_program_dims)(C.c_void_p(handle), out), "tz_program_dims")
    return tuple(int(v) for v in out[:7])


def last_error() -> str:
    buf = C.create_string_buffer(512)
    lib().tz_last_error(buf, 512)
    return buf.value.decode(errors="replace")


def check(rc: int, what: str) -> None:
    if rc != TZ_OK:
        raise RuntimeError(f"{what} failed (code {rc}): {last_error()}")


def _host(a, dtype) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, dtype=dtype))


_DESC_ARRAYS = ("P", "q0", "Qp", "A", "l0", "u0", "kink0", "wabs", "R", "Bt", "gam", "Rchk", "cc", "CC2", "XB", "ze1_val", "D", "E", "K")


def _describe(L, handle, obj):
    """bucket name, warm rows and tube pattern of a program handle -> attributes of obj"""
    buf = C.create_string_buffer(64)
    L.tz_program_bucket(handle, buf, 64)
    obj.bucket = buf.value.decode()
    obj.warm_rows = int(L.tz_program_warm_rows(handle))
    nnz = int(L.tz_program_tube_pattern(handle, None, 0))
    pat = np.zeros(max(nnz, 1), dtype=np.int32)
    L.tz_program_tube_pattern(handle, pat.ctypes.data, nnz)
    obj.tube_pattern = pat[:nnz]           # row-major indices of the entries of Ze[1].Z that are not structurally zero


class Program:
    """Owner of a TzProgram handle built from a tzddpc_b200.program.CompiledProgram."""

    def __init__(self, prog, K: np.ndarray):
        L = lib()
        order = np.argsort(-(prog.wabs > 0).astype(np.int64), kind="stable")       # |.|-cost rows first
        f64 = lambda a: _host(a, np.float64)                                        # noqa: E731
        A, l0, u0 = f64(prog.A[order]), f64(prog.l0[order]), f64(prog.u0[order])
        kink0, wabs, R, E = f64(prog.kink0[order]), f64(prog.wabs[order]), f64(prog.R[order]), f64(prog.E[order])
        arrs = dict(P=f64(prog.P), q0=f64(prog.q0), Qp=f64(prog.Qp), A=A, l0=l0, u0=u0, kink0=kink0, wabs=wabs, R=R,
                    Bt=f64(prog.Bt), gam=f64(prog.gam), Rchk=f64(prog.Rchk), cc=f64(prog.cc), CC2=f64(prog.CC2),
                    XB=f64(prog.XB), ze1_ptr=_host(prog.ze1_ptr, np.int32), ze1_idx=_host(prog.ze1_idx, np.int32),
                    ze1_val=f64(prog.ze1_val), D=f64(prog.D), E=E, K=f64(K))
        d = TzProgramDesc()
        d.n, d.m, d.horizon, d.nv, d.nz, d.nc = prog.n, prog.m, prog.N, prog.nv, prog.nz, prog.nc
        d.npar, d.na, d.nchk, d.nkink = prog.npar, prog.na, prog.Rchk.shape[0], int((prog.wabs > 0).sum())
        d.g1, d.nterms, d.c = prog.g1, len(prog.ze1_idx), float(prog.c)
        for k, a in arrs.items():
            setattr(d, k, a.ctypes.data if a.size else None)
        h = C.c_void_p()
        check(L.tz_program_create(C.byref(d), C.byref(h)), "tz_program_create")
        self.handle = h
        self.row_order = order
        self.compiled = prog
        _describe(L, h, self)

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                lib().tz_program_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class ProgramView:
    """Program d of a ProgramBatch: the interface of Program (handle, compiled, bucket, ...), borrowed from the batch."""

    def __init__(self, batch: "ProgramBatch", d: int, handle):
        self._batch, self._d, self.handle = batch, d, handle
        self.row_order, self.bucket, self.warm_rows, self.tube_pattern = batch.row_order, batch.bucket, batch.warm_rows, batch.tube_pattern
        self._compiled = None

    @property
    def compiled(self):
        if self._compiled is None:
            self._compiled = self._batch.compiled.program(self._d)
        return self._compiled


class ProgramBatch:
    """Owner of a TzProgramBatch: the D programs of a tzddpc_b200.program.CompiledProgramBatch (one per data set), packed on
    the host and uploaded with one copy.  `programs[d]` behaves like a Program."""

    def __init__(self, cbatch, K: np.ndarray):
        L = lib()
        D = cbatch.num
        order = np.argsort(-(cbatch.wabs[0] > 0).astype(np.int64), kind="stable")   # |.|-cost rows first (the structure is shared)
        f64 = lambda a: _host(a, np.float64)                                        # noqa: E731
        K = np.broadcast_to(np.asarray(K, dtype=np.float64).reshape((-1, cbatch.m, cbatch.n)), (D, cbatch.m, cbatch.n))
        arrs = dict(P=f64(cbatch.P), q0=f64(cbatch.q0), Qp=f64(cbatch.Qp), A=f64(cbatch.A[:, order]), l0=f64(cbatch.l0[:, order]),
                    u0=f64(cbatch.u0[:, order]), kink0=f64(cbatch.kink0[:, order]), wabs=f64(cbatch.wabs[:, order]),
                    R=f64(cbatch.R[:, order]), Bt=f64(cbatch.Bt), gam=f64(cbatch.gam), Rchk=f64(cbatch.Rchk), cc=f64(cbatch.cc),
                    CC2=f64(cbatch.CC2), XB=f64(cbatch.XB), ze1_val=f64(cbatch.ze1_val), D=f64(cbatch.D_), E=f64(cbatch.E[:, order]), K=f64(K))
        ptr, idx = _host(cbatch.ze1_ptr, np.int32), _host(cbatch.ze1_idx, np.int32)
        descs = (TzProgramDesc * D)()
        nkink = int((cbatch.wabs[0] > 0).sum())
        base = {k: (a.ctypes.data, a[0].nbytes if a.size else 0, a.size) for k, a in arrs.items()}
        for d in range(D):
            t = descs[d]
            t.n, t.m, t.horizon, t.nv, t.nz, t.nc = cbatch.n, cbatch.m, cbatch.N, cbatch.nv, cbatch.nz, cbatch.nc
            t.npar, t.na, t.nchk, t.nkink = cbatch.npar, cbatch.na, cbatch.Rchk.shape[1], nkink
            t.g1, t.nterms, t.c = cbatch.g1, len(idx), float(cbatch.c[d])
            for k in _DESC_ARRAYS:
                p0, stride, size = base[k]
                setattr(t, k, p0 + d * stride if size else None)
            t.ze1_ptr, t.ze1_idx = ptr.ctypes.data, (idx.ctypes.data if idx.size else None)
        h = C.c_void_p()
        check(L.tz_program_create_batch(descs, D, C.byref(h)), "tz_program_create_batch")
        self.handle, self.compiled, self.row_order, self.num = h, cbatch, order, D
        h0 = C.c_void_p(L.tz_program_batch_get(h, 0))
        _describe(L, h0, self)
        self.programs = [ProgramView(self, d, C.c_void_p(L.tz_program_batch_get(h, d))) for d in range(D)]

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                lib().tz_program_batch_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class ProgramSet:
    """Owner of a TzProgramSet: D programs of one structure (one per data set), scenarios [begin[j], begin[j+1]) use program j."""

    def __init__(self, programs, begin):
        L = lib()
        self.programs = list(programs)                      # keeps the borrowed handles alive
        self.begin = np.ascontiguousarray(np.asarray(begin, dtype=np.int64))
        assert len(self.begin) == len(self.programs) + 1
        arr = (C.c_void_p * len(self.programs))(*[p.handle.value for p in self.programs])
        h = C.c_void_p()
        check(L.tz_program_set_create(arr, len(self.programs), self.begin.ctypes.data, C.byref(h)), "tz_program_set_create")
        self.handle = h
        self.scenarios = int(self.begin[-1])

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                lib().tz_program_set_destroy(self.handle)
                self.handle = None
        except Exception:
            pass
