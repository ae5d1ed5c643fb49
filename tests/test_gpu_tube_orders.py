"""The fused tube rollout beyond the orders whose pre-reduction block fits in shared memory (order 31 at n = 5):
tz_tube_rollout then runs tube_rollout_recompute_kernel, which evaluates the block's columns where the Girard passes read
them.  Checked against the oracle applied stepwise, against the chain of stand-alone kernels, bit for bit against the
resident kernel (TZDDPC_ROLLOUT) wherever both fit, for writes outside its outputs, at its order limit and at the
262,144 scenarios of BASELINE.json configs[4]."""
import ctypes as C

import numpy as np
import pytest
import torch

from tests import common
from tests.test_gpu_guard_bands import Guarded
from tests.test_gpu_tube import _model, _oracle_rollout

pytestmark = pytest.mark.gpu

METRICS = {"l1-linf": 0, "l1": 1, "l2": 2}


def f(a):
    return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def _gcap(n, order):
    return int(np.floor(n * (order - 1))) + n


def _inputs(seed, S, steps, n=5, m=1):
    rng = np.random.default_rng(seed)
    Z0 = np.zeros((S, n, 2)); Z0[:, :, 0] = rng.uniform(-0.3, 0.3, size=(S, n))      # Ze[0] = <e0, zeros(n, 1)>
    XU = rng.uniform(-2, 2, size=(S, steps, n + m))
    return Z0, XU


def _rollout(monkeypatch, kernel, *args):
    if kernel is None:
        monkeypatch.delenv("TZDDPC_ROLLOUT", raising=False)
    else:
        monkeypatch.setenv("TZDDPC_ROLLOUT", kernel)
    out = torch.ops.tzddpc.tube_rollout(*args)
    torch.cuda.synchronize()
    monkeypatch.delenv("TZDDPC_ROLLOUT", raising=False)
    return out


def _check_oracle(Zf, gf, lo, hi, models, Z0, XU, order, metric):
    Zf, gf, lo, hi = Zf.cpu().numpy(), gf.cpu().numpy(), lo.cpu().numpy(), hi.cpu().numpy()
    for s in range(Z0.shape[0]):
        A, GK, GD, W = models[s]
        Zo, hulls = _oracle_rollout(A, GK, GD, W, Z0[s], XU[s], order, metric)
        for k in range(XU.shape[1]):
            np.testing.assert_allclose(lo[s, k], hulls[k].left_limit, rtol=common.GEN_RTOL, atol=1e-12)
            np.testing.assert_allclose(hi[s, k], hulls[k].right_limit, rtol=common.GEN_RTOL, atol=1e-12)
        assert gf[s] == Zo.num_generators
        np.testing.assert_allclose(Zf[s, :, 0], Zo.center, rtol=common.GEN_RTOL, atol=1e-12)
        np.testing.assert_allclose(Zf[s, :, 1:1 + gf[s]], Zo.generators, rtol=1e-8, atol=1e-12)      # same columns, same order
        assert not np.any(Zf[s, :, 1 + gf[s]:])


@pytest.mark.parametrize("order,steps,metric,boxed", [(32, 4, "l1-linf", True), (40, 4, "l2", True), (40, 3, "l1", False),
                                                      (60, 3, "l1-linf", False), (60, 4, "l1", True), (120, 3, "l2", False),
                                                      (120, 4, "l1-linf", True)])
def test_recompute_rollout_matches_oracle(cuda_lib, monkeypatch, order, steps, metric, boxed):
    """Forced to the recompute kernel: with the 7 + 6 generators of the dense model the resident block still fits at
    orders 40 and 60."""
    from tzddpc_b200 import ops  # noqa: F401
    n, m, S = 5, 1, 4
    A, GK, GD, W = _model(order * 7 + steps, n, m, boxed)
    Z0, XU = _inputs(steps, S, steps)
    Zf, gf, lo, hi = _rollout(monkeypatch, "recompute", f(A), f(GK), f(GD), f(Z0), f(XU), f(W), float(order), METRICS[metric],
                              _gcap(n, order))
    assert int(gf.min()) > 5 * (order - 1)          # reduced at the last step
    _check_oracle(Zf, gf, lo, hi, [(A, GK, GD, W)] * S, Z0, XU, order, metric)


def test_recompute_rollout_per_scenario_model_matches_oracle(cuda_lib, monkeypatch):
    from tzddpc_b200 import ops  # noqa: F401
    n, m, S, order, steps = 5, 1, 4, 40, 3
    models = [_model(100 + s, n, m, s % 2 == 0) for s in range(S)]
    nk = max(M[1].shape[0] for M in models)          # pad the boxed / dense generator lists to one count with zero matrices
    nd = max(M[2].shape[0] for M in models)
    CK = np.stack([M[0] for M in models])
    GK = np.zeros((S, nk, n, n)); GD = np.zeros((S, nd, n, n + m))
    for s, M in enumerate(models):
        GK[s, :M[1].shape[0]] = M[1]; GD[s, :M[2].shape[0]] = M[2]
    W = models[0][3]
    Z0, XU = _inputs(9, S, steps)
    Zf, gf, lo, hi = _rollout(monkeypatch, "recompute", f(CK), f(GK), f(GD), f(Z0), f(XU), f(W), float(order), 0, _gcap(n, order))
    _check_oracle(Zf, gf, lo, hi, [(CK[s], GK[s], GD[s], W) for s in range(S)], Z0, XU, order, "l1-linf")


def test_recompute_rollout_equals_chain_of_standalone_kernels(cuda_lib):
    """Order 40: the recompute kernel against reach_step -> girard_reduce -> interval_hull."""
    n, m, S, order, steps = 5, 1, 64, 40.0, 6
    A, GK, GD, W = _model(3, n, m, True)
    Z0, XU = _inputs(1, S, steps)
    gcap = _gcap(n, order)
    Zf, gf, lo, hi = torch.ops.tzddpc.tube_rollout(f(A), f(GK), f(GD), f(Z0), f(XU), f(W), order, 0, gcap)
    Z = f(Z0)
    zeroC = f(np.zeros((n, n + m)))
    for k in range(steps):
        T1 = torch.ops.tzddpc.reach_step(f(A), f(GK), Z, None)
        xu = torch.zeros((S, n + m, 2), dtype=torch.float64, device="cuda")
        xu[:, :, 0] = f(XU[:, k])
        Zn = torch.ops.tzddpc.reach_step(zeroC, f(GD), xu, f(W))
        pre = torch.cat([T1, Zn[:, :, 1:]], dim=2)
        pre[:, :, 0] += Zn[:, :, 0]
        red, gout = torch.ops.tzddpc.girard_reduce(pre.contiguous(), order, 0, gcap)
        g = int(gout.max().item())
        Z = red[:, :, :1 + g].contiguous()
        l2, h2 = torch.ops.tzddpc.interval_hull(Z)
        torch.testing.assert_close(lo[:, k], l2, rtol=1e-10, atol=1e-12)
        torch.testing.assert_close(hi[:, k], h2, rtol=1e-10, atol=1e-12)
    assert int(gf.min()) == gcap
    torch.testing.assert_close(Zf[:, :, :Z.shape[2]], Z, rtol=1e-9, atol=1e-12)


def _assert_kernels_equal(monkeypatch, args):
    a = _rollout(monkeypatch, "resident", *args)
    b = _rollout(monkeypatch, "recompute", *args)
    for x, y, what in zip(a, b, ("Zfinal", "gfinal", "hull_lo", "hull_hi")):
        assert torch.equal(x, y), what
    return a


@pytest.mark.parametrize("metric", [0, 1, 2])
@pytest.mark.parametrize("order", [2, 5, 10, 20, 30, 31])
def test_recompute_equals_resident_bit_for_bit(cuda_lib, monkeypatch, order, metric):
    """Wherever both kernels fit they compute the same bits: the same products, keys, selection, box and hull.  Some
    entries of z_k are zero, so that some columns of the block are zero generators."""
    n, m, S, steps = 5, 1, 16, 4
    A, GK, GD, W = _model(order + 11 * metric, n, m, order % 2 == 0)
    Z0, XU = _inputs(order, S, steps)
    XU[::3, :, 2] = 0.0
    XU[1::4, 1:, :] = 0.0
    _assert_kernels_equal(monkeypatch, (f(A), f(GK), f(GD), f(Z0), f(XU), f(W), float(order), metric, _gcap(n, order)))


@pytest.mark.parametrize("metric", [0, 1, 2])
def test_recompute_equals_resident_with_equal_keys(cuda_lib, monkeypatch, metric):
    """A boxed model with equal box entries: many generators share their key, so the ties-by-lowest-index path runs."""
    n, m, S, steps, order = 5, 1, 16, 4, 10
    A, GK, GD, W = _model(5, n, m, True)
    GK[GK != 0] = 0.01; GD[GD != 0] = 0.01
    Z0, XU = _inputs(5, S, steps)
    XU[:, :, :] = np.round(XU * 2) / 2                 # few distinct magnitudes in z_k
    _assert_kernels_equal(monkeypatch, (f(A), f(GK), f(GD), f(Z0), f(XU), f(W), float(order), metric, _gcap(n, order)))


@pytest.mark.parametrize("metric", [0, 1, 2])
def test_recompute_equals_resident_with_large_g0(cuda_lib, monkeypatch, metric):
    """g0 = 40 generators in Z0, above the 10 that the reduction at order 2 leaves."""
    n, m, S, steps, order, g0 = 5, 1, 16, 3, 2, 40
    A, GK, GD, W = _model(6, n, m, False)
    rng = np.random.default_rng(6)
    Z0 = rng.uniform(-0.3, 0.3, size=(S, n, 1 + g0)); Z0[:, :, 7] = 0.0
    _, XU = _inputs(6, S, steps)
    Zf, gf, _, _ = _assert_kernels_equal(monkeypatch, (f(A), f(GK), f(GD), f(Z0), f(XU), f(W), float(order), metric, g0))
    assert int(gf.max()) == _gcap(n, order)


@pytest.mark.parametrize("metric", [0, 1, 2])
def test_recompute_equals_resident_when_gcap_is_too_small(cuda_lib, monkeypatch, metric):
    """At order 1.2, n = 5: floor(5 (1.2 - 1)) + 5 = 5 is the smallest gcap accepted, but 5 * 1.2 rounds to 6.0, so six
    non-zero generators are not reduced.  M_K with one zero generator, one generator of M_Delta and no W leave exactly
    g + 1 non-zero columns: the step writes 6 into a gcap of 5 and reports the truncation (negative gfinal)."""
    n, m, S, steps, order, g0 = 5, 1, 8, 3, 1.2, 5
    A, _, GD, _ = _model(7, n, m, False)
    GK = np.zeros((1, n, n))
    rng = np.random.default_rng(7)
    Z0 = rng.uniform(-0.3, 0.3, size=(S, n, 1 + g0))
    _, XU = _inputs(7, S, steps)
    Zf, gf, _, _ = _assert_kernels_equal(monkeypatch, (f(A), f(GK), f(GD[:1]), f(Z0), f(XU), None, order, metric, g0))
    assert bool((gf == -g0).all())


@pytest.mark.parametrize("kernel", ["resident", "recompute"])
def test_rollout_sizes_its_block_for_generators_kept_by_rounding(cuda_lib, monkeypatch, kernel):
    """Order 1.2, n = 5, gcap = 6: floor(5 (1.2 - 1)) + 5 = 5, but 5 * 1.2 rounds to 6.0, so a step keeps 6 generators
    unreduced and the next step's block has (NK + 1) * 6 + ... columns, more than a block sized for 5.  Both kernels
    against the oracle (1, 2 and 3 steps: 6, 5 and 6 generators)."""
    n, m, S, steps, order, g0 = 5, 1, 8, 3, 1.2, 5
    A, _, GD, _ = _model(7, n, m, False)
    GK, W = np.zeros((1, n, n)), np.zeros((n, 2))
    rng = np.random.default_rng(7)
    Z0 = rng.uniform(-0.3, 0.3, size=(S, n, 1 + g0))
    _, XU = _inputs(7, S, steps)
    Zf, gf, lo, hi = _rollout(monkeypatch, kernel, f(A), f(GK), f(GD[:1]), f(Z0), f(XU), f(W), order, 0, 6)
    assert bool((gf == 6).all())
    _check_oracle(Zf, gf, lo, hi, [(A, GK, GD[:1], W)] * S, Z0, XU, order, "l1-linf")


def test_recompute_rollout_stays_inside_its_buffers(cuda_lib):
    """Order 40 through the C ABI, every output a window of a sentinel-filled allocation: the kernel alternates between two
    zonotopes in shared memory and must write Zfinal, gfinal and the hulls and nothing around them."""
    from tzddpc_b200 import _abi
    n, m, S, steps, order = 5, 1, 37, 4, 40.0
    A, GK, GD, W = _model(8, n, m, True)
    Z0, XU = _inputs(8, S, steps)
    gcap = _gcap(n, order)
    dev = torch.device("cuda")
    gb = Guarded(dev)
    Zf = gb.make((S, n, 1 + gcap))
    gf = gb.make((S,), dtype=torch.int32)
    lo = gb.make((S, steps, n))
    hi = gb.make((S, steps, n))
    ins = [f(A), f(GK), f(GD), f(Z0), f(XU), f(W)]
    p = lambda t: C.c_void_p(t.data_ptr())      # noqa: E731
    rc = _abi.lib().tz_tube_rollout(S, n, m, GK.shape[0], GD.shape[0], W.shape[1] - 1, 1, steps, order, 0, p(ins[0]), p(ins[1]),
                                    p(ins[2]), 0, p(ins[3]), p(ins[4]), p(ins[5]), gcap, p(Zf), p(gf), p(lo), p(hi),
                                    C.c_void_p(torch.cuda.current_stream().cuda_stream))
    _abi.check(rc, "tz_tube_rollout")
    torch.cuda.synchronize()
    gb.check("tube_rollout order 40")
    assert bool((gf == gcap).all())
    assert bool(torch.isfinite(lo).all()) and bool(torch.isfinite(hi).all())
    ref = torch.ops.tzddpc.tube_rollout(*ins[:6], order, 0, gcap)
    for x, y in zip(ref, (Zf, gf, lo, hi)):
        assert torch.equal(x, y)


def test_recompute_order_limit(cuda_lib, monkeypatch):
    """n = 5, m = 1, 25 + 30 + 1 generators of M_K, M_Delta and W: order 135 (17,606 columns before reduction, 225,006 bytes
    of shared memory) is the largest that runs; order 136 (226,576 bytes) is rejected with both sizes.  TZDDPC_ROLLOUT cannot
    force the resident kernel where it does not fit, and takes no other values."""
    n, m, S, steps = 5, 1, 2, 3
    A, GK, GD, W = _model(10, n, m, True)
    Z0, XU = _inputs(10, S, steps)
    args = lambda order: (f(A), f(GK), f(GD), f(Z0), f(XU), f(W), float(order), 0, _gcap(n, order))      # noqa: E731
    Zf, gf, lo, hi = torch.ops.tzddpc.tube_rollout(*args(135))
    assert bool((gf == _gcap(n, 135)).all()) and bool(torch.isfinite(hi).all())
    with pytest.raises(RuntimeError, match=r"17736 generators before reduction\) needs \d+ bytes .* and 226576 with it recomputed"):
        torch.ops.tzddpc.tube_rollout(*args(136))
    with pytest.raises(RuntimeError, match=r"needs \d+ bytes of shared memory with the block resident"):
        _rollout(monkeypatch, "resident", *args(40))
    with pytest.raises(RuntimeError, match="TZDDPC_ROLLOUT must be resident or recompute"):
        _rollout(monkeypatch, "fused", *args(10))


def test_recompute_rollout_at_scale(cuda_lib):
    """BASELINE.json configs[4] at order 40: 262,144 scenarios, every one reduced to 200 generators with a finite hull, and
    64 seeded scenarios give the same bits in a batch of their own."""
    n, m, S, steps, order = 5, 1, 262144, 4, 40.0
    A, GK, GD, W = _model(0, n, m, True)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(40)
    Z0 = torch.zeros((S, n, 2), dtype=torch.float64, device="cuda")
    Z0[:, :, 0] = torch.rand((S, n), dtype=torch.float64, device="cuda", generator=gen) - 0.5
    XU = torch.rand((S, steps, n + m), dtype=torch.float64, device="cuda", generator=gen) * 4 - 2
    gcap = _gcap(n, order)
    model = (f(A), f(GK), f(GD))
    Zf, gf, lo, hi = torch.ops.tzddpc.tube_rollout(*model, Z0, XU, f(W), order, 0, gcap)
    assert bool((gf == 200).all())
    assert bool(torch.isfinite(lo).all()) and bool(torch.isfinite(hi).all())
    pick = torch.as_tensor(np.sort(np.random.default_rng(64).choice(S, 64, replace=False)), device="cuda")
    Zs, gs, ls, hs = torch.ops.tzddpc.tube_rollout(*model, Z0[pick].contiguous(), XU[pick].contiguous(), f(W), order, 0, gcap)
    assert torch.equal(Zs, Zf[pick]) and torch.equal(gs, gf[pick]) and torch.equal(ls, lo[pick]) and torch.equal(hs, hi[pick])
