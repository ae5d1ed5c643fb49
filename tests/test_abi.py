"""The C ABI without a GPU: libtzddpc.so builds (nvcc cross-compiles sm_100a), loads, exports exactly the
functions include/tzddpc.h declares, and its host-only entry points behave.  No compute call is made here."""
import ctypes as C
import os
import re
import subprocess
from pathlib import Path

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "tzddpc.h")


def declared_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(tz_[a-z0-9_]+)\s*\(", src)))


def test_header_declares_what_the_binding_lists():
    from tzddpc_b200 import _abi
    assert declared_functions() == sorted(_abi.EXPORTS)


def test_library_exports_every_declared_symbol(cuda_lib):
    for name in declared_functions():
        assert hasattr(cuda_lib, name), f"libtzddpc.so does not export {name}"


def test_library_is_sm100a_and_self_contained(cuda_lib):
    from tzddpc_b200 import _abi, build
    cuobjdump = Path(build._nvcc()).with_name("cuobjdump")       # the toolkit that built the library, whether on PATH or not
    if not cuobjdump.exists():
        pytest.skip("cuobjdump not available")
    out = subprocess.run([str(cuobjdump), "--list-elf", str(_abi.LIB_PATH)], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert "sm_100a" in out.stdout
    ldd = subprocess.run(["ldd", str(_abi.LIB_PATH)], capture_output=True, text=True).stdout
    assert "libtorch" not in ldd and "libcudart" not in ldd        # plain C ABI, static CUDA runtime


def test_host_only_entry_points(cuda_lib):
    from tzddpc_b200 import _abi
    assert b"tzddpc-b200" in cuda_lib.tz_version()
    o = _abi.TzSolverOpts()
    cuda_lib.tz_solver_opts_default(C.byref(o))
    assert o.rho > 0 and 0 < o.alpha < 2 and o.max_iter >= 100 and o.eps_abs == pytest.approx(1e-6)
    # argument validation happens before any CUDA call and reports through tz_last_error
    rc = cuda_lib.tz_program_create(None, None)
    assert rc == -22
    assert "null" in _abi.last_error()
    assert cuda_lib.tz_program_warm_rows(None) == -22
    assert cuda_lib.tz_closed_loop_step_host_scratch_bytes(None, 10) == 0


def test_struct_layouts_match_the_header(cuda_lib):
    """ctypes mirrors of TzProgramDesc / TzSolverOpts: field order and sizes as in include/tzddpc.h."""
    from tzddpc_b200 import _abi
    assert C.sizeof(_abi.TzSolverOpts) == 88          # 7 doubles + 7 int32, padded to 8
    names = [f[0] for f in _abi.TzProgramDesc._fields_]
    src = open(HEADER).read()
    body = src[src.index("typedef struct TzProgramDesc {"):src.index("} TzProgramDesc;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    decl = []
    for stmt in body.split("{", 1)[1].split(";"):
        stmt = stmt.strip()
        if not stmt:
            continue
        stmt = re.sub(r"^(const\s+)?(int32_t|double)\s*", "", stmt)
        decl += [t.strip().lstrip("*").strip() for t in stmt.split(",")]
    assert decl == names


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    from tzddpc_b200 import _abi
    monkeypatch.setattr(_abi, "_lib", None)
    monkeypatch.setattr(_abi, "LIB_PATH", tmp_path / "nope.so")
    with pytest.raises(_abi.TzddpcLibraryMissing, match="no CPU fallback"):
        _abi.lib()


def test_controller_refuses_to_run_without_a_gpu():
    import numpy as np
    import torch
    import tzddpc_b200 as tz
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        tz.TZDDPC(tz.Data(np.zeros((10, 1)), np.zeros((10, 2))))


def test_public_names_mirror_the_reference_package():
    """tzddpc/__init__.py:1-15 re-exports; tzddpc/tzddpc.py public methods and properties."""
    import tzddpc_b200 as tz
    for name in ("TZDDPC", "Data", "SystemZonotopes", "Theta", "DataDrivenDataset", "OptimizationProblem",
                 "OptimizationProblemVariables"):
        assert hasattr(tz, name)
    for meth in ("update_identification_data", "build_zonotopes", "compute_theta", "build_zonotopes_theta",
                 "build_problem", "build_problem_simplified", "solve", "num_samples", "dim_u", "dim_x"):
        assert hasattr(tz.TZDDPC, meth)
    assert tz.Data._fields == ("u", "x") and tz.SystemZonotopes._fields == ("X0", "U", "X", "W")
    assert tz.Theta._fields == ("K", "deltaA", "deltaB")
    for name in ("compute_theta", "compute_A_B", "compute_control_gain", "spectral_radius"):      # tzddpc/__init__.py:2-7
        assert callable(getattr(tz, name))
    import numpy as np
    assert tz.spectral_radius(np.array([[0.5, 1.0], [0.0, -0.8]])) == 0.8
