"""BASELINE.json configs[4] (synthetic 5-dim system, long horizon, high zonotope order): the fused tube rollout
Z_{k+1} = reduce(M_K x Z_k + M_Delta x <[xbar_k; v_k], 0> + W, order) against the oracle applied stepwise
(oracle MatrixZonotope * Zonotope, Minkowski sums, Zonotope.reduce), and against the chain of the stand-alone
kernels reach_step -> girard_reduce -> interval_hull."""
import numpy as np
import pytest

import oracle
from tests import common
from tzddpc_b200 import configs

pytestmark = pytest.mark.gpu


def _model(seed, n=5, m=1, boxed=True):
    rng = np.random.default_rng(seed)
    A = rng.normal(size=(n, n))
    A *= 0.85 / np.abs(np.linalg.eigvals(A)).max()                 # Schur-stable closed loop centre
    if boxed:       # order-1 boxed M_K / M_Delta as build_zonotopes_theta leaves them (single-entry generators)
        dK = rng.uniform(0.001, 0.02, size=(n, n))
        dD = rng.uniform(0.001, 0.02, size=(n, n + m))
        GK = np.zeros((n * n, n, n)); GD = np.zeros((n * (n + m), n, n + m))
        for r in range(n):
            for c in range(n):
                GK[r * n + c, r, c] = dK[r, c]
            for c in range(n + m):
                GD[r * (n + m) + c, r, c] = dD[r, c]
    else:
        GK = 0.02 * rng.normal(size=(7, n, n)); GD = 0.02 * rng.normal(size=(6, n, n + m))
    W = np.hstack([np.zeros((n, 1)), 0.1 * np.ones((n, 1))])
    return A, GK, GD, W


def _oracle_rollout(A, GK, GD, W, Z0, XU, order, metric):
    conv = oracle.Conventions(girard_metric=metric)
    n = A.shape[0]
    W = np.zeros((n, 1)) if W is None else W                                    # no noise: W = <0, no generators>
    MK = oracle.MatrixZonotope(A, GK, conv)
    MD = oracle.MatrixZonotope(np.zeros(GD.shape[1:]), GD, conv)                # (GD may hold no generator)
    Wz = oracle.Zonotope(W[:, 0], W[:, 1:], conv)
    Z = oracle.Zonotope(Z0[:, 0], Z0[:, 1:], conv)
    hulls = []
    for k in range(XU.shape[0]):
        zk = oracle.Zonotope(XU[k], np.zeros((XU.shape[1], 1)), conv)            # <[xbar_k; v_k], 0>  (tzddpc/tzddpc.py:174)
        Z = ((MK * Z) + ((MD * zk) + Wz)).reduce(order)                          # :175-176,185,205 + reduce
        hulls.append(Z.interval)
    return Z, hulls


@pytest.mark.parametrize("order,steps,metric,boxed", [(2, 6, "l1-linf", True), (5, 8, "l1-linf", True), (10, 5, "l2", True),
                                                      (3, 6, "l1", False), (20, 3, "l1-linf", True)])
def test_tube_rollout_matches_oracle(cuda_lib, order, steps, metric, boxed):
    import torch
    from tzddpc_b200 import ops  # noqa: F401
    n, m, S = 5, 1, 6
    A, GK, GD, W = _model(order * 7 + steps, n, m, boxed)
    rng = np.random.default_rng(steps)
    Z0 = np.zeros((S, n, 2)); Z0[:, :, 0] = rng.uniform(-0.3, 0.3, size=(S, n))      # Ze[0] = <e0, zeros(n, 1)>  (:172)
    XU = rng.uniform(-2, 2, size=(S, steps, n + m))
    gcap = int(np.floor(n * (order - 1))) + n
    f = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).cuda()    # noqa: E731
    mid = {"l1-linf": 0, "l1": 1, "l2": 2}[metric]
    Zf, gf, lo, hi = torch.ops.tzddpc.tube_rollout(f(A), f(GK), f(GD), f(Z0), f(XU), f(W), float(order), mid, gcap)
    Zf, gf, lo, hi = Zf.cpu().numpy(), gf.cpu().numpy(), lo.cpu().numpy(), hi.cpu().numpy()
    for s in range(S):
        Zo, hulls = _oracle_rollout(A, GK, GD, W, Z0[s], XU[s], order, metric)
        for k in range(steps):       # the interval hull is invariant under the choice of the boxed generators
            np.testing.assert_allclose(lo[s, k], hulls[k].left_limit, rtol=common.GEN_RTOL, atol=1e-12)
            np.testing.assert_allclose(hi[s, k], hulls[k].right_limit, rtol=common.GEN_RTOL, atol=1e-12)
        assert gf[s] == Zo.num_generators
        np.testing.assert_allclose(Zf[s, :, 0], Zo.center, rtol=common.GEN_RTOL, atol=1e-12)
        np.testing.assert_allclose(Zf[s, :, 1:1 + gf[s]], Zo.generators, rtol=1e-8, atol=1e-12)      # same columns, same order
        assert not np.any(Zf[s, :, 1 + gf[s]:])


def test_tube_rollout_equals_chain_of_standalone_kernels(cuda_lib):
    """Two independent CUDA paths: the fused rollout and reach_step -> girard_reduce -> interval_hull."""
    import torch
    n, m, S, order, steps = 5, 1, 64, 4.0, 4
    A, GK, GD, W = _model(3, n, m, True)
    rng = np.random.default_rng(1)
    Z0 = np.zeros((S, n, 2)); Z0[:, :, 0] = rng.uniform(-0.3, 0.3, size=(S, n))
    XU = rng.uniform(-2, 2, size=(S, steps, n + m))
    gcap = int(np.floor(n * (order - 1))) + n
    f = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).cuda()    # noqa: E731
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
    torch.testing.assert_close(Zf[:, :, :Z.shape[2]], Z, rtol=1e-9, atol=1e-12)


def test_tube_rollout_first_step_is_the_reference_tube(cuda_lib):
    """With order = infinity-like (no reduction needed) one rollout step from Ze[0] = <e0, 0> reproduces the set Ze[1]
    that `solve` returns (same generators up to the zero columns the reduction drops)."""
    import torch
    cfg = configs.pulley()
    u, x = common.dataset(cfg)
    o, K = common.make_oracle(cfg, u, x)
    n, m = cfg.n, cfg.m
    rng = np.random.default_rng(2)
    e0 = rng.uniform(-0.2, 0.2, n); xb = 1.0 + rng.uniform(-0.2, 0.2, n); v = np.array([0.3, 0.1])
    Ze1 = o.evaluate_tube(xb, e0, v, 1)
    f = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).cuda()    # noqa: E731
    Z0 = np.zeros((1, n, 2)); Z0[0, :, 0] = e0
    XU = np.r_[xb, v[0]][None, None]
    Zf, gf, lo, hi = torch.ops.tzddpc.tube_rollout(f(o.MdataK.center), f(o.MdataK.generators), f(o.Mdelta.generators), f(Z0), f(XU),
                                                   f(o.zonotopes.W.Z), 20.0, 0, 80)      # 75 generators <= 20 * 4: no reduction
    G = Ze1[:, 1:]
    Gnz = G[:, np.any(G != 0, axis=0)]
    g = int(gf[0])
    assert g == Gnz.shape[1]
    np.testing.assert_allclose(Zf[0, :, 0].cpu().numpy(), Ze1[:, 0], rtol=common.GEN_RTOL, atol=1e-12)
    np.testing.assert_allclose(common.sort_columns(Zf[0, :, 1:1 + g].cpu().numpy()), common.sort_columns(Gnz), rtol=common.GEN_RTOL, atol=1e-13)
