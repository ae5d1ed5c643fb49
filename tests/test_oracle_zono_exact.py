"""The references of tests/test_gpu_zono_dims.py, checked without a GPU: on that file's exact inputs (entries k/16) the
oracle (oracle/zono.py: matzono_times_Z, girard_reduce_generators, Zonotope.interval, and the stepwise tube rollout of
tests/test_gpu_tube.py) equals the exact rational computation with fractions.Fraction value for value, so that those
inputs really stay exact and the GPU file may compare bit for bit.  Also the exact-product helper of its rounding bounds
against Fraction."""
from fractions import Fraction

import numpy as np
import pytest

import oracle
from oracle.zono import girard_reduce_generators, matzono_times_Z
from tests import test_gpu_zono_dims as Z
from tests.test_gpu_tube import _oracle_rollout


def _equal(a, q):
    """float array a equals the Fraction array q exactly (value for value)."""
    return a.shape == q.shape and bool(np.all(Z.Q(a) == q))


@pytest.mark.parametrize("case", Z.REACH_CASES, ids=Z.reach_id)
def test_reach_oracle_is_exact(case):
    n, p, N, g, gW, per = case
    Cm, Gm, Zin, W = Z.reach_inputs(case)
    for s in range(Zin.shape[0]):
        q = Z.q_product(Cm[s] if per else Cm, Gm[s] if per else Gm, Zin[s])
        if W is not None:
            q = np.hstack([q, Z.Q(W[:, 1:])])
            q[:, 0] += Z.Q(W[:, 0])
        assert _equal(Z.reach_oracle(Cm, Gm, Zin, W, s, per), q)


def test_largest_matrix_zonotope_oracle_is_exact():
    """The largest case of test_reach_step_largest_matrix_zonotope (N = 2132 matrices 3 x 4)."""
    rng = np.random.default_rng(2132)
    Cm, Zin = Z.dyadic(rng, (3, 4)), Z.dyadic(rng, (1, 4, 3))
    Gm = Z.dyadic(rng, (2133, 3, 4))[:2132]
    assert _equal(matzono_times_Z(Cm, Gm, Zin[0]), Z.q_product(Cm, Gm, Zin[0]))


@pytest.mark.parametrize("case", Z.GIRARD_CASES, ids=Z.girard_id)
def test_girard_oracle_is_exact(case):
    n, g, order = case
    Zin = Z.girard_inputs(n, g)
    for metric in Z.NAMES:
        for s in range(Zin.shape[0]):
            ref = girard_reduce_generators(Zin[s, :, 1:], order, oracle.Conventions(girard_metric=metric))
            assert _equal(ref, Z.q_girard(Z.Q(Zin[s, :, 1:]), order, metric)), (metric, s)


@pytest.mark.parametrize("n", Z.HULL_DIMS)
def test_interval_oracle_is_exact(n):
    for g in Z.HULL_GENS:
        Zin = Z.hull_inputs(n, g)
        for s in range(Zin.shape[0]):
            iv = oracle.Zonotope(Zin[s, :, 0], Zin[s, :, 1:]).interval
            lo, hi = Z.q_interval(Z.Q(Zin[s]))
            assert _equal(iv.left_limit, lo) and _equal(iv.right_limit, hi), g


def _oracle_steps(A, GK, GD, W, Z0, XU, order, metric):
    """_oracle_rollout with every intermediate kept: (pre-reduction Z, reduced Z, hull lo, hull hi) per step."""
    conv = oracle.Conventions(girard_metric=metric)
    n = A.shape[0]
    W = np.zeros((n, 1)) if W is None else W
    MK = oracle.MatrixZonotope(A, GK, conv)
    MD = oracle.MatrixZonotope(np.zeros(GD.shape[1:]), GD, conv)
    Wz = oracle.Zonotope(W[:, 0], W[:, 1:], conv)
    Zc = oracle.Zonotope(Z0[:, 0], Z0[:, 1:], conv)
    out = []
    for k in range(XU.shape[0]):
        zk = oracle.Zonotope(XU[k], np.zeros((XU.shape[1], 1)), conv)
        pre = (MK * Zc) + ((MD * zk) + Wz)
        Zc = pre.reduce(order)
        out.append((pre.Z, Zc.Z, Zc.interval.left_limit, Zc.interval.right_limit))
    return out


@pytest.mark.parametrize("case", [c for c in Z.ROLLOUT_CASES if min(Z.rollout_inputs(c)["sizes"][1:]) <= Z.ROLLOUT_SMEM],
                         ids=Z.rollout_id)
def test_rollout_oracle_is_exact_at_every_step(case):
    """Every rollout case that a kernel runs: each intermediate of the oracle's rollout equals its Fraction counterpart,
    and the oracle rollout the GPU file compares with ends where these steps end."""
    d = Z.rollout_inputs(case)
    for s in range(d["Z0"].shape[0]):
        args = (*d["models"][s], d["Z0"][s], d["XU"][s], d["order"], d["metric"])
        steps = _oracle_steps(*args)
        qsteps = Z.q_rollout(*args)
        for k, (fl, q) in enumerate(zip(steps, qsteps)):
            for what, a, b in zip(("pre-reduction", "reduced", "hull lo", "hull hi"), fl, q):
                assert _equal(a, b), (s, k, what)
        Zo, hulls = _oracle_rollout(*args)
        assert np.array_equal(Zo.Z, steps[-1][1]) and all(np.array_equal(h.left_limit, st[2]) for h, st in zip(hulls, steps))


def test_rollout_cases_reach_every_kernel_and_the_size_limit():
    """The ids of the rollout cases name resident and recompute runs at m >= 2 and n > 8, recompute-only runs (the
    controller's largest system, n = 8, m = 4 boxed at order 5, among them) and cases where neither kernel fits."""
    ids = [Z.rollout_id(c) for c in Z.ROLLOUT_CASES]
    both = [i for i in ids if i.endswith("resident+recompute")]
    assert any("-m2-" in i or "-m4-" in i for i in both) and any(int(i.split("-")[0][1:]) > 8 for i in both)
    assert "n8-m4-boxed-order5-shared-recompute" in ids
    assert any(i.endswith("neither-fits") for i in ids)
    assert any(i.startswith("n16-m2-dense-order10") and i.endswith("-recompute") for i in ids)


def test_exact_products_helper_against_fractions():
    rng = np.random.default_rng(0)
    M = rng.normal(size=(3, 7)) * 10.0 ** rng.integers(-8, 8, size=(3, 7))
    X = rng.normal(size=(7, 5))
    got = Z.exact_fsum_products(M, X)
    q = Z.Q(M).dot(Z.Q(X))
    assert all(got.flat[i] == float(q.flat[i]) for i in range(got.size))
    assert all(isinstance(x, Fraction) for x in q.flat)
