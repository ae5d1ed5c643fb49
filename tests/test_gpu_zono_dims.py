"""The stand-alone zonotope kernels and the fused tube rollout of tz_zono.cu at every dimension and dispatch branch:
reach_kernel_fast (the six TZ_FAST pairs), reach_kernel<8> (n <= 8), reach_kernel<16> (9 <= n <= 16), girard_warp_kernel
(g <= 128 and n <= 8), girard_kernel (n > 8 or g > 128, up to n = 128), hull_kernel, and tube_rollout_kernel /
tube_rollout_recompute_kernel (resident where the 220 KiB of shared memory hold the pre-reduction block, recomputed
otherwise) at n = 1-16 and m = 1, 2, 4.

Two kinds of reference:
* exact inputs: entries k/16 (small |k|), so that every product and sum of these shapes is exact in fp64.  The kernels'
  results are then exact whatever their FMA contraction or summation order, the oracle's are too, Girard selection is the
  same on both sides and equal metrics are real ties.  Compared bit for bit, which catches any indexing, chunking or
  column-map error whatever its size.  tests/test_oracle_zono_exact.py proves on the CPU, against fractions.Fraction, that
  these inputs do stay exact.
* random real inputs: against the exact value (Fraction / math.fsum) within a rigorous rounding bound
  (gamma_k = k u / (1 - k u) times the sum of the magnitudes), and the two rollout kernels against each other bitwise.

Also the shapes reach_step / tube_rollout refuse before any launch (their C entry points take raw pointers)."""
import ctypes as C
import math
from fractions import Fraction

import numpy as np
import pytest
import torch

import oracle
from oracle.zono import girard_reduce_generators, matzono_times_Z
from tests.test_gpu_guard_bands import Guarded
from tests.test_gpu_tube import _model, _oracle_rollout

pytestmark = pytest.mark.gpu

U = 2.0 ** -53                                   # unit roundoff of fp64
METRICS = {"l1-linf": 0, "l1": 1, "l2": 2}
NAMES = list(METRICS)
FAST = [(2, 2), (2, 3), (4, 4), (4, 5), (5, 5), (5, 6)]     # TZ_FAST pairs (n, p) of tz_reach_step
ROLLOUT_SMEM = 220 * 1024                         # shared memory a tube rollout may use


def gamma(k):
    return k * U / (1.0 - k * U)


def f(a):
    return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def dyadic(rng, shape, k=15):
    """Entries j/16 with |j| <= k."""
    return rng.integers(-k, k + 1, size=shape) / 16.0


# ---- exact rational reference ---------------------------------------------------------------------------------------
def Q(a):
    """float64 array -> object array of the same values as Fractions (exact)."""
    a = np.asarray(a, dtype=np.float64)
    return np.array([Fraction(x) for x in a.flat] + [None], dtype=object)[:-1].reshape(a.shape)


def q_product(Cm, Gm, Z):
    """Exact [C Z, G_1 Z, ..., G_N Z] (the column order of matzono_times_Z)."""
    Zq = Q(Z)
    return np.concatenate([Q(Cm).dot(Zq)] + [Q(G).dot(Zq) for G in Gm], axis=1)


def q_metric(a, metric):
    if metric == "l1-linf":
        return [sum(a[:, j]) - max(a[:, j]) for j in range(a.shape[1])]
    if metric == "l1":
        return [sum(a[:, j]) for j in range(a.shape[1])]
    return [sum(x * x for x in a[:, j]) for j in range(a.shape[1])]


def q_girard(G, order, metric):
    """Exact Girard reduction of a Fraction generator block: zero columns dropped; if more than order * n remain, the
    g - floor(n (order - 1)) of smallest exact metric (ties: lowest index) are boxed into diag(sum |.|)."""
    n = G.shape[0]
    G = G[:, [j for j in range(G.shape[1]) if any(x != 0 for x in G[:, j])]]
    g = G.shape[1]
    if g <= order * n:
        return G
    n_red = g - int(math.floor(n * (order - 1)))
    a = np.abs(G)
    h = q_metric(a, metric)
    idx = sorted(range(g), key=lambda j: (h[j], j))
    red, keep = sorted(idx[:n_red]), sorted(idx[n_red:])
    box = np.full((n, n), Fraction(0), dtype=object)
    for r in range(n):
        box[r, r] = sum(a[r, red])
    return np.hstack([G[:, keep], box])


def q_interval(Z):
    d = np.array([sum(abs(x) for x in Z[r, 1:]) for r in range(Z.shape[0])] + [None], dtype=object)[:-1]
    return Z[:, 0] - d, Z[:, 0] + d


def q_rollout(A, GK, GD, W, Z0, XU, order, metric):
    """_oracle_rollout in exact arithmetic: per step (pre-reduction zonotope, reduced zonotope, hull lo, hull hi), with
    the oracle's column order (zero columns of M_Delta x <z_k, 0> included)."""
    n, p = A.shape[0], XU.shape[1]
    W = np.zeros((n, 1)) if W is None else W
    Wq = Q(W)
    Z = Q(Z0)
    out = []
    for k in range(XU.shape[0]):
        T = q_product(A, GK, Z)
        D = q_product(np.zeros((n, p)), GD, np.c_[XU[k], np.zeros(p)])
        pre = np.hstack([(T[:, :1] + (D[:, :1] + Wq[:, :1])), T[:, 1:], D[:, 1:], Wq[:, 1:]])
        Z = np.hstack([pre[:, :1], q_girard(pre[:, 1:], order, metric)])
        out.append((pre, Z) + q_interval(Z))
    return out


def exact_fsum_products(M, Z):
    """M @ Z correctly rounded: every product split exactly into two doubles (Veltkamp / Dekker), summed by math.fsum."""
    def split(a):
        t = a * 134217729.0
        hi = t - (t - a)
        return hi, a - hi
    P = M[:, :, None] * Z[None, :, :]
    mh, ml = split(M[:, :, None] + 0 * Z[None])
    zh, zl = split(Z[None] + 0 * M[:, :, None])
    E = ((mh * zh - P) + mh * zl + ml * zh) + ml * zl
    out = np.empty((M.shape[0], Z.shape[1]))
    for r in range(M.shape[0]):
        for j in range(Z.shape[1]):
            out[r, j] = math.fsum(np.r_[P[r, :, j], E[r, :, j]])
    return out


# ---- cases ----------------------------------------------------------------------------------------------------------
def _reach_branch(n, p):
    return f"fast{n}x{p}" if (n, p) in FAST else ("reach8" if n <= 8 else "reach16")


# (n, p, N, g, gW, per-scenario model); gW = -1: no W, gW = 0: a W with a centre and no generator
REACH_CASES = [(2, 2, 4, 3, 1, False), (2, 3, 3, 5, 0, True), (4, 4, 16, 7, 1, False), (4, 5, 20, 2, 2, True),
               (5, 5, 25, 1, -1, False), (5, 6, 30, 1, 1, False)]
REACH_CASES += [(5, 6, 3, g, 1, False) for g in (0, 31, 32, 255, 256)]          # 1+g = 1, 32, 33, 256, 257 column threads
REACH_CASES += [(1, 3, 2, 5, 1, False), (1, 1, 0, 4, 0, False), (6, 4, 3, 9, 2, True), (7, 9, 2, 40, -1, False),
                (8, 8, 5, 31, 0, False), (8, 3, 4, 256, 1, True), (3, 2, 0, 0, 1, False)]
REACH_CASES += [(9, 5, 3, 6, 1, False), (12, 14, 2, 33, 0, True), (16, 16, 3, 32, 2, False), (16, 20, 1, 256, 1, False),
                (16, 9, 0, 10, -1, False)]


def reach_id(c):
    n, p, N, g, gW, per = c
    return f"{_reach_branch(n, p)}-n{n}-p{p}-N{N}-g{g}-gW{gW if gW >= 0 else 'none'}-{'per' if per else 'shared'}"


def reach_inputs(c, S=3):
    n, p, N, g, gW, per = c
    rng = np.random.default_rng(1009 * n + 97 * p + 13 * N + g)
    Cm = dyadic(rng, (S, n, p) if per else (n, p))
    Gm = dyadic(rng, (S, N, n, p) if per else (N, n, p))
    Z = dyadic(rng, (S, p, 1 + g))
    W = None if gW < 0 else dyadic(rng, (n, 1 + gW))
    return Cm, Gm, Z, W


def reach_oracle(Cm, Gm, Z, W, s, per):
    ref = matzono_times_Z(Cm[s] if per else Cm, Gm[s] if per else Gm, Z[s])
    if W is not None:                  # Minkowski sum with W (tzddpc/tzddpc.py:176)
        ref = np.hstack([ref, W[:, 1:]])
        ref[:, 0] += W[:, 0]
    return ref


def _girard_branch(n, g):
    return "warp" if g <= 128 and n <= 8 else "cta"


GIRARD_CASES = [(n, g, 2.5) for n in range(1, 9) for g in (127, 128)]            # girard_warp_kernel, n = 1..8
GIRARD_CASES += [(n, 129, 2.5) for n in (1, 5, 8)]                               # girard_kernel just above g = 128
GIRARD_CASES += [(n, 3 * n + 7, o) for n in (9, 16, 17, 64, 96, 128) for o in (1, 1.5, 2, 2.7)]      # n > 8: 8-row chunks
GIRARD_CASES += [(3, 300, 2.7), (9, 600, 1.5), (17, 1100, 2.0)]                  # g > 256, > 512: multi-column ranges


def girard_id(c):
    n, g, order = c
    return f"{_girard_branch(n, g)}-n{n}-g{g}-order{order}"


def girard_inputs(n, g, S=3, seed=0):
    """Scenario 0 plain, 1 with zero and -0.0 columns, 2 with its second half a copy of the first (exact ties)."""
    rng = np.random.default_rng(seed + 7 * n + g)
    Z = dyadic(rng, (S, n, 1 + g))
    Z[1, :, 1 + 3::7] = 0.0
    Z[1, :, 1 + 5::11] = -0.0
    if S > 2:
        Z[2, :, 1 + g // 2:] = Z[2, :, 1:1 + (g - g // 2)]
    return Z


def girard_cap(n, g, order):
    return max(g, int(np.ceil(n * order)) + n)


HULL_DIMS = list(range(1, 17)) + [128]
HULL_GENS = (0, 31, 32, 33, 1000)


def hull_inputs(n, g, S=3):
    rng = np.random.default_rng(31 * n + g)
    return dyadic(rng, (S, n, 1 + g))


def rollout_smem(n, m, NK, ND, gW, g0, order, gcap):
    """(generators before reduction, resident bytes, recompute bytes) as tz_tube_rollout sizes its two kernels."""
    gred = int(math.floor(n * (order - 1))) + n
    gmax = max(g0, gred)
    gkeep = int(math.floor(n * order))
    gstep = min(gkeep, gcap) if gkeep > gmax else gmax
    gpre = (NK + 1) * gstep + NK + ND + gW
    p = n + m
    res = (n * (1 + gcap) + n * gpre + (NK + 1) * n * n + ND * n * p + p + n + 2) * 8 + gpre * 9 + 16
    rc = (2 * n * (1 + gcap) + (NK + 1) * n * n + ND * n * p + p + 1) * 8 + gpre * 9 + 16
    return gpre, res, rc


def exact_model(rng, n, m, kind):
    """Boxed: single-entry generators as build_zonotopes_theta leaves M_K / M_Delta; dense: 7 + 6 full generators."""
    p = n + m
    A = dyadic(rng, (n, n), 4)
    if kind == "boxed":
        GK = np.zeros((n * n, n, n)); GD = np.zeros((n * p, n, p))
        for r in range(n):
            for c in range(n):
                GK[r * n + c, r, c] = rng.integers(1, 4) / 16.0
            for c in range(p):
                GD[r * p + c, r, c] = rng.integers(1, 4) / 16.0
    else:
        GK = dyadic(rng, (7, n, n), 3); GD = dyadic(rng, (6, n, p), 3)
    W = dyadic(rng, (n, 3))
    return A, GK, GD, W


# (n, m, boxed / dense, order, variant): boxed at order 2, dense at order 5, and the larger orders named in the ids
ROLLOUT_CASES = [(n, m, k, 2 if k == "boxed" else 5, "shared") for n in (1, 2, 3, 7, 8, 9, 12, 16) for m in (1, 2, 4)
                 for k in ("boxed", "dense")]
ROLLOUT_CASES += [(8, 4, "boxed", 5, "shared"), (16, 2, "dense", 10, "shared"), (16, 4, "dense", 10, "per"),
                  (3, 2, "dense", 5, "per"), (9, 4, "dense", 5, "per"), (8, 2, "boxed", 2, "per"), (7, 2, "dense", 5, "noW"),
                  (12, 4, "dense", 5, "noW"), (2, 4, "dense", 5, "NK0"), (9, 1, "dense", 5, "NK0"), (3, 1, "boxed", 2, "ND0"),
                  (16, 2, "dense", 5, "ND0"), (1, 4, "boxed", 10, "NK0")]
ROLLOUT_STEPS, ROLLOUT_S = 3, 2


def rollout_inputs(case):
    """Exact inputs of a rollout case: models[s] = (CK, GK, GD, W) of scenario s, the op's arguments and the sizes."""
    n, m, kind, order, variant = case
    rng = np.random.default_rng(7919 * n + 131 * m + 17 * order + 3 * len(variant) + (kind == "boxed"))
    S, steps, p = ROLLOUT_S, ROLLOUT_STEPS, n + m
    ms = [exact_model(rng, n, m, kind) for _ in range(S if variant == "per" else 1)]
    ms = [(A, GK, GD, ms[0][3]) for A, GK, GD, _ in ms]          # W is shared by the scenarios
    if variant == "noW":
        ms = [(A, GK, GD, None) for A, GK, GD, _ in ms]
    if variant == "NK0":
        ms = [(A, GK[:0], GD, W) for A, GK, GD, W in ms]
    if variant == "ND0":
        ms = [(A, GK, GD[:0], W) for A, GK, GD, W in ms]
    Z0 = dyadic(rng, (S, n, 3))
    XU = dyadic(rng, (S, steps, p))
    XU[0, 1, ::2] = 0.0                                  # zero entries of z_k: zero columns of M_Delta x z_k
    per = variant == "per"
    CK = np.stack([M[0] for M in ms]) if per else ms[0][0]
    GK = np.stack([M[1] for M in ms]) if per else ms[0][1]
    GD = np.stack([M[2] for M in ms]) if per else ms[0][2]
    W = ms[0][3]
    gcap = int(math.floor(n * (order - 1))) + n
    metric = NAMES[(n + m + int(order)) % 3]
    models = [ms[s] if per else ms[0] for s in range(S)]
    gW = 0 if W is None else W.shape[1] - 1
    sizes = rollout_smem(n, m, GK.shape[-3], GD.shape[-3], gW, Z0.shape[2] - 1, order, gcap)
    return dict(models=models, CK=CK, GK=GK, GD=GD, W=W, Z0=Z0, XU=XU, order=float(order), metric=metric, gcap=gcap, sizes=sizes)


def rollout_id(case):
    n, m, kind, order, variant = case
    d = rollout_inputs(case)
    _, res, rc = d["sizes"]
    fits = "+".join(k for k, b in (("resident", res), ("recompute", rc)) if b <= ROLLOUT_SMEM) or "neither-fits"
    return f"n{n}-m{m}-{kind}-order{order}-{variant}-{fits}"


# ---- reach_step -----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def T(cuda_lib):
    from tzddpc_b200 import ops  # noqa: F401  (registers torch.ops.tzddpc)
    return torch


@pytest.mark.parametrize("case", REACH_CASES, ids=reach_id)
def test_reach_step_exact(T, case):
    n, p, N, g, gW, per = case
    Cm, Gm, Z, W = reach_inputs(case)
    out = T.ops.tzddpc.reach_step(f(Cm), f(Gm), f(Z), None if W is None else f(W)).cpu().numpy()
    assert out.shape == (Z.shape[0], n, (N + 1) * (1 + g) + max(gW, 0))
    for s in range(Z.shape[0]):
        np.testing.assert_array_equal(out[s], reach_oracle(Cm, Gm, Z, W, s, per))


@pytest.mark.parametrize("case", [(2, 3, 4, 40, 1, True), (5, 6, 30, 255, 1, False), (3, 4, 5, 10, 2, False),
                                  (8, 6, 3, 100, 0, True), (9, 12, 4, 60, 1, False), (16, 16, 2, 256, 1, True)], ids=reach_id)
def test_reach_step_random_within_rounding_bound(T, case):
    """|gpu - exact| <= gamma_p sum_k |M_rk| |z_kj| (+ the centre's one addition of W), the exact product by fsum."""
    n, p, N, g, gW, per = case
    rng = np.random.default_rng(n * p + g)
    S = 2
    Cm = rng.normal(size=(S, n, p) if per else (n, p))
    Gm = rng.normal(size=(S, N, n, p) if per else (N, n, p)) * rng.uniform(0.01, 10, size=(N, 1, 1))
    Z = rng.normal(size=(S, p, 1 + g))
    W = rng.normal(size=(n, 1 + gW))
    out = T.ops.tzddpc.reach_step(f(Cm), f(Gm), f(Z), f(W)).cpu().numpy()
    for s in range(S):
        Ms = [Cm[s] if per else Cm] + list(Gm[s] if per else Gm)
        exact = np.hstack([exact_fsum_products(M, Z[s]) for M in Ms])
        mag = np.hstack([np.abs(M) @ np.abs(Z[s]) for M in Ms])
        bound = gamma(p + 1) * mag * (1 + 4 * gamma(p))
        bound[:, 0] += 2 * U * (np.abs(exact[:, 0]) + np.abs(W[:, 0]))
        exact[:, 0] += W[:, 0]
        got = out[s, :, :exact.shape[1]]
        assert np.all(np.abs(got - exact) <= bound), np.max(np.abs(got - exact) / np.maximum(bound, 1e-300))
        np.testing.assert_array_equal(out[s, :, exact.shape[1]:], W[:, 1:])


@pytest.mark.parametrize("n,p,kernel", [(5, 6, "fast5x6"), (8, 8, "reach8"), (3, 4, "reach8"), (16, 16, "reach16")])
def test_reach_step_largest_matrix_zonotope(T, n, p, kernel):
    """The largest N whose (N+1) staged matrices fit the 200 KiB of shared memory runs (bitwise against the oracle); N + 1
    is refused.  The fast path stages its matrices with the rows padded to an even count."""
    rows = n + (n & 1) if kernel.startswith("fast") else n
    N = 200 * 1024 // (rows * p * 8) - 1
    rng = np.random.default_rng(N)
    Cm, Z = dyadic(rng, (n, p)), dyadic(rng, (1, p, 3))
    Gm = dyadic(rng, (N + 1, n, p))
    out = T.ops.tzddpc.reach_step(f(Cm), f(Gm[:N]), f(Z), None).cpu().numpy()
    np.testing.assert_array_equal(out[0], matzono_times_Z(Cm, Gm[:N], Z[0]))
    with pytest.raises(RuntimeError, match="matrix zonotope too large for shared memory"):
        T.ops.tzddpc.reach_step(f(Cm), f(Gm), f(Z), None)


# ---- girard_reduce --------------------------------------------------------------------------------------------------
def _check_girard(out, gout, Z, order, metric):
    n = Z.shape[1]
    for s in range(Z.shape[0]):
        ref = girard_reduce_generators(Z[s, :, 1:], order, oracle.Conventions(girard_metric=metric))
        assert gout[s] == ref.shape[1], (metric, s, gout[s], ref.shape)
        np.testing.assert_array_equal(out[s, :, 0], Z[s, :, 0])
        np.testing.assert_array_equal(out[s, :, 1:1 + gout[s]], ref, err_msg=f"{metric} scenario {s} (n={n})")
        assert not np.any(out[s, :, 1 + gout[s]:])


@pytest.mark.parametrize("case", GIRARD_CASES, ids=girard_id)
def test_girard_reduce_exact(T, case):
    n, g, order = case
    Z = girard_inputs(n, g)
    for metric in NAMES:
        out, gout = T.ops.tzddpc.girard_reduce(f(Z), order, METRICS[metric], girard_cap(n, g, order))
        _check_girard(out.cpu().numpy(), gout.cpu().numpy(), Z, order, metric)


@pytest.mark.parametrize("g", [100, 300], ids=["warp-n1-g100", "cta-n1-g300"])
def test_girard_reduce_one_dimension_is_all_ties(T, g):
    """n = 1, l1-linf: every metric is |x| - |x| = 0, so the selection is ties only (the lowest indices are reduced)."""
    Z = girard_inputs(1, g)
    out, gout = T.ops.tzddpc.girard_reduce(f(Z), 3.0, 0, girard_cap(1, g, 3.0))
    out, gout = out.cpu().numpy(), gout.cpu().numpy()
    _check_girard(out, gout, Z, 3.0, "l1-linf")
    nz = np.flatnonzero(Z[0, 0, 1:] != 0)
    np.testing.assert_array_equal(out[0, 0, 1:3], Z[0, 0, 1 + nz[-2:]])         # the two highest-index columns are kept


@pytest.mark.parametrize("kernel,n,g,order,cap", [("warp", 5, 100, 2.0, 7), ("cta", 12, 300, 2.0, 15), ("warp", 4, 20, 8.0, 9),
                                                  ("cta", 3, 200, 1.0, 2)])
def test_girard_reduce_cap_too_small(T, kernel, n, g, order, cap):
    """gout_cap below the generator count: gout = -count, the first cap columns as the oracle's, and nothing written outside
    Zout / gout (every output a window of a sentinel-filled allocation, through the C ABI)."""
    from tzddpc_b200 import _abi
    assert (kernel == "warp") == (g <= 128 and n <= 8)
    S = 3
    Z = girard_inputs(n, g, S, seed=cap)
    dev = torch.device("cuda")
    gb = Guarded(dev)
    out = gb.make((S, n, 1 + cap))
    gout = gb.make((S,), dtype=torch.int32)
    Zd = f(Z)
    p = lambda t: C.c_void_p(t.data_ptr())      # noqa: E731
    for metric in NAMES:
        rc = _abi.lib().tz_girard_reduce(S, n, g, order, METRICS[metric], p(Zd), cap, p(out), p(gout),
                                         C.c_void_p(torch.cuda.current_stream().cuda_stream))
        _abi.check(rc, "tz_girard_reduce")
        torch.cuda.synchronize()
        gb.check(f"{kernel} n={n} g={g} cap={cap} {metric}")
        o, go = out.cpu().numpy(), gout.cpu().numpy()
        for s in range(S):
            ref = girard_reduce_generators(Z[s, :, 1:], order, oracle.Conventions(girard_metric=metric))
            assert ref.shape[1] > cap and go[s] == -ref.shape[1], (s, go[s], ref.shape)
            np.testing.assert_array_equal(o[s, :, 0], Z[s, :, 0])
            np.testing.assert_array_equal(o[s, :, 1:], ref[:, :cap])


def test_girard_reduce_rejects_n_129(T):
    with pytest.raises(RuntimeError, match=r"n <= 128"):
        T.ops.tzddpc.girard_reduce(f(np.ones((1, 129, 400))), 2.0, 0, 400)


@pytest.mark.parametrize("n", [2, 5, 8])
def test_girard_warp_compensated_box(T, n):
    """Kept columns carry ~2^40 in every row, reduced ones ~1: girard_warp_kernel computes the box as (sum of all) - (sum
    of the kept) with Neumaier compensation, and must land within a few ulps of the exact reduced sum.  The plain
    difference of the two rounded sums would be off by ~1e-3 relative."""
    g, order, S = 120, 4.0, 4
    rng = np.random.default_rng(n)
    Z = rng.uniform(-1, 1, size=(S, n, 1 + g))
    big = np.sort(rng.choice(g, int(n * (order - 1)), replace=False))
    Z[:, :, 1 + big] = 2.0 ** 40 * rng.uniform(0.5, 1.0, size=(S, n, len(big))) * rng.choice([-1, 1], size=(S, n, len(big)))
    for metric in NAMES:
        out, gout = T.ops.tzddpc.girard_reduce(f(Z), order, METRICS[metric], girard_cap(n, g, order))
        out, gout = out.cpu().numpy(), gout.cpu().numpy()
        red = np.setdiff1d(np.arange(g), big)
        for s in range(S):
            kept = len(big)
            assert gout[s] == kept + n
            np.testing.assert_array_equal(out[s, :, 1:1 + kept], Z[s][:, 1 + big])
            box = out[s, :, 1 + kept:1 + kept + n]
            exact = np.array([math.fsum(np.abs(Z[s, r, 1 + red])) for r in range(n)])
            np.testing.assert_array_equal(box - np.diag(np.diag(box)), 0.0)
            err = np.abs(np.diag(box) - exact)
            assert np.all(err <= 8 * np.spacing(exact)), (metric, s, err / np.spacing(exact))


@pytest.mark.parametrize("n,g", [(3, 129), (9, 300), (17, 1100), (128, 600)], ids=lambda v: str(v))
def test_girard_cta_box_within_rounding_bound(T, n, g):
    """girard_kernel on random reals: the selection is the oracle's (kept columns bitwise) and every box entry is within
    gamma_g sum |g_red| of the exact sum over the reduced columns."""
    order, S = 2.0, 2
    rng = np.random.default_rng(g)
    Z = rng.normal(size=(S, n, 1 + g)) * rng.uniform(1e-3, 1e3, size=(S, 1, 1 + g))
    for metric in NAMES:
        out, gout = T.ops.tzddpc.girard_reduce(f(Z), order, METRICS[metric], girard_cap(n, g, order))
        out, gout = out.cpu().numpy(), gout.cpu().numpy()
        for s in range(S):
            ref = girard_reduce_generators(Z[s, :, 1:], order, oracle.Conventions(girard_metric=metric))
            kept = ref.shape[1] - n
            assert gout[s] == ref.shape[1]
            np.testing.assert_array_equal(out[s, :, 1:1 + kept], ref[:, :kept])
            keep_idx = [int(np.flatnonzero((Z[s, :, 1:] == ref[:, j:j + 1]).all(axis=0))[0]) for j in range(kept)]
            red = np.setdiff1d(np.arange(g), keep_idx)
            exact = np.array([math.fsum(np.abs(Z[s, r, 1 + red])) for r in range(n)])
            err = np.abs(np.diag(out[s, :, 1 + kept:1 + kept + n]) - exact)
            assert np.all(err <= gamma(len(red)) * exact), (metric, s)


# ---- interval_hull --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", HULL_DIMS)
def test_interval_hull_exact(T, n):
    for g in HULL_GENS:
        Z = hull_inputs(n, g)
        lo, hi = T.ops.tzddpc.interval_hull(f(Z))
        for s in range(Z.shape[0]):
            iv = oracle.Zonotope(Z[s, :, 0], Z[s, :, 1:]).interval
            np.testing.assert_array_equal(lo[s].cpu().numpy(), iv.left_limit, err_msg=f"g={g}")
            np.testing.assert_array_equal(hi[s].cpu().numpy(), iv.right_limit, err_msg=f"g={g}")


@pytest.mark.parametrize("n,g", [(3, 1000), (16, 33), (128, 999)])
def test_interval_hull_within_rounding_bound(T, n, g):
    rng = np.random.default_rng(n + g)
    Z = rng.normal(size=(2, n, 1 + g)) * rng.uniform(1e-3, 1e3, size=(2, 1, 1 + g))
    lo, hi = T.ops.tzddpc.interval_hull(f(Z))
    lo, hi = lo.cpu().numpy(), hi.cpu().numpy()
    for s in range(2):
        A = np.array([math.fsum(np.abs(Z[s, r, 1:])) for r in range(n)])
        c = Z[s, :, 0]
        for got, sign in ((lo[s], -1), (hi[s], 1)):
            exact = np.array([float(Fraction(c[r]) + sign * Fraction(A[r])) for r in range(n)])
            assert np.all(np.abs(got - exact) <= gamma(g) * A + 2 * U * np.abs(exact))


# ---- tube_rollout ---------------------------------------------------------------------------------------------------
def _rollout(monkeypatch, kernel, *args):
    if kernel is None:
        monkeypatch.delenv("TZDDPC_ROLLOUT", raising=False)
    else:
        monkeypatch.setenv("TZDDPC_ROLLOUT", kernel)
    try:
        out = torch.ops.tzddpc.tube_rollout(*args)
        torch.cuda.synchronize()
    finally:
        monkeypatch.delenv("TZDDPC_ROLLOUT", raising=False)
    return out


def _rollout_args(d):
    return (f(d["CK"]), f(d["GK"]), f(d["GD"]), f(d["Z0"]), f(d["XU"]), None if d["W"] is None else f(d["W"]), d["order"],
            METRICS[d["metric"]], d["gcap"])


def _chain(d):
    """reach_step -> girard_reduce -> interval_hull per step, as in tests/test_gpu_tube.py, per-scenario models included."""
    CK, GK, GD, W = f(d["CK"]), f(d["GK"]), f(d["GD"]), None if d["W"] is None else f(d["W"])
    Z0, XU = d["Z0"], d["XU"]
    S, steps, p = XU.shape
    zeroC = torch.zeros(tuple(d["CK"].shape[:-1]) + (p,), dtype=torch.float64, device="cuda")
    Z, hulls = f(Z0), []
    for k in range(steps):
        T1 = torch.ops.tzddpc.reach_step(CK, GK, Z, None)
        xu = torch.zeros((S, p, 2), dtype=torch.float64, device="cuda")
        xu[:, :, 0] = f(XU[:, k])
        Zn = torch.ops.tzddpc.reach_step(zeroC, GD, xu, W)
        pre = torch.cat([T1, Zn[:, :, 1:]], dim=2)
        pre[:, :, 0] += Zn[:, :, 0]
        red, gout = torch.ops.tzddpc.girard_reduce(pre.contiguous(), d["order"], METRICS[d["metric"]], d["gcap"])
        Z = red[:, :, :1 + int(gout.max().item())].contiguous()
        hulls.append(torch.ops.tzddpc.interval_hull(Z))
    return Z, gout, hulls


def _chain_fits(d):
    n, p = d["Z0"].shape[1], d["XU"].shape[2]
    NK, ND = d["GK"].shape[-3], d["GD"].shape[-3]
    return (NK + 1) * n * n * 8 <= 200 * 1024 and (ND + 1) * n * p * 8 <= 200 * 1024


def _oracle(d):
    return [_oracle_rollout(*d["models"][s], d["Z0"][s], d["XU"][s], d["order"], d["metric"]) for s in range(d["Z0"].shape[0])]


def _check_rollout_exact(out, ref):
    Zf, gf, lo, hi = (x.cpu().numpy() for x in out)
    for s, (Zo, hulls) in enumerate(ref):
        for k, iv in enumerate(hulls):
            np.testing.assert_array_equal(lo[s, k], iv.left_limit, err_msg=f"scenario {s} step {k}")
            np.testing.assert_array_equal(hi[s, k], iv.right_limit, err_msg=f"scenario {s} step {k}")
        assert gf[s] == Zo.num_generators
        np.testing.assert_array_equal(Zf[s, :, 0], Zo.center)
        np.testing.assert_array_equal(Zf[s, :, 1:1 + gf[s]], Zo.generators)
        assert not np.any(Zf[s, :, 1 + gf[s]:])


@pytest.mark.parametrize("case", ROLLOUT_CASES, ids=rollout_id)
def test_tube_rollout_exact(T, monkeypatch, case):
    """Each kernel that fits (forced with TZDDPC_ROLLOUT) and the default dispatch bitwise against the oracle stepwise
    and against the chain of stand-alone kernels; a kernel that does not fit raises naming both sizes."""
    n = case[0]
    d = rollout_inputs(case)
    gpre, res, rc = d["sizes"]
    args = _rollout_args(d)
    msg = rf"\(n={n}, {gpre} generators before reduction\) needs {res} bytes of shared memory .* and {rc} with it recomputed"
    outs, ref = [], _oracle(d) if min(res, rc) <= ROLLOUT_SMEM else None
    for kernel, need in (("resident", res), ("recompute", rc), (None, min(res, rc))):
        if need <= ROLLOUT_SMEM:
            outs.append(_rollout(monkeypatch, kernel, *args))
            _check_rollout_exact(outs[-1], ref)
        else:
            with pytest.raises(RuntimeError, match=msg):
                _rollout(monkeypatch, kernel, *args)
    for o in outs[1:]:
        assert all(torch.equal(x, y) for x, y in zip(outs[0], o))
    if outs and _chain_fits(d):
        Z, gout, hulls = _chain(d)
        Zf, gf, lo, hi = outs[0]
        for k, (l2, h2) in enumerate(hulls):
            assert torch.equal(lo[:, k], l2) and torch.equal(hi[:, k], h2), k
        assert torch.equal(gf, gout)
        assert torch.equal(Zf[:, :, :Z.shape[2]], Z)


RANDOM_ROLLOUTS = [(1, 2, False, 5), (3, 4, True, 5), (7, 2, True, 2), (8, 4, True, 2), (9, 2, False, 10), (12, 4, False, 5),
                   (16, 1, False, 5), (16, 4, False, 2), (2, 1, True, 10)]


@pytest.mark.parametrize("n,m,boxed,order", RANDOM_ROLLOUTS,
                         ids=[f"n{n}-m{m}-{'boxed' if b else 'dense'}-order{o}" for n, m, b, o in RANDOM_ROLLOUTS])
def test_rollout_kernels_agree_bitwise_on_random_inputs(T, monkeypatch, n, m, boxed, order):
    """Resident and recompute compute the same bits wherever both fit, at every metric; some entries of z_k are zero."""
    A, GK, GD, W = _model(n * 10 + m, n, m, boxed)
    S, steps = 8, 3
    rng = np.random.default_rng(n + m)
    Z0 = np.zeros((S, n, 2)); Z0[:, :, 0] = rng.uniform(-0.3, 0.3, size=(S, n))
    XU = rng.uniform(-2, 2, size=(S, steps, n + m))
    XU[::3, :, 1] = 0.0
    gcap = int(math.floor(n * (order - 1))) + n
    _, res, rc = rollout_smem(n, m, GK.shape[0], GD.shape[0], 1, 1, order, gcap)
    assert res <= ROLLOUT_SMEM and rc <= ROLLOUT_SMEM
    for metric in range(3):
        args = (f(A), f(GK), f(GD), f(Z0), f(XU), f(W), float(order), metric, gcap)
        a = _rollout(monkeypatch, "resident", *args)
        b = _rollout(monkeypatch, "recompute", *args)
        for x, y, what in zip(a, b, ("Zfinal", "gfinal", "hull_lo", "hull_hi")):
            assert torch.equal(x, y), (what, metric)


def test_rollout_at_the_controllers_largest_system(T, monkeypatch):
    """n = 8, m = 4 with boxed M_K / M_Delta (64 + 96 generators, as build_zonotopes_theta leaves them) at order 5: the
    resident block does not fit, the default dispatch runs the recompute kernel, against the oracle stepwise."""
    from tests import common
    n, m, order, S, steps = 8, 4, 5.0, 16, 4
    A, GK, GD, W = _model(84, n, m, True)
    gcap = int(math.floor(n * (order - 1))) + n
    _, res, rc = rollout_smem(n, m, GK.shape[0], GD.shape[0], 1, 1, order, gcap)
    assert res > ROLLOUT_SMEM >= rc
    rng = np.random.default_rng(84)
    Z0 = np.zeros((S, n, 2)); Z0[:, :, 0] = rng.uniform(-0.3, 0.3, size=(S, n))
    XU = rng.uniform(-2, 2, size=(S, steps, n + m))
    Zf, gf, lo, hi = (x.cpu().numpy() for x in _rollout(monkeypatch, None, f(A), f(GK), f(GD), f(Z0), f(XU), f(W), order, 0, gcap))
    assert (gf == gcap).all()
    for s in range(0, S, 5):
        Zo, hulls = _oracle_rollout(A, GK, GD, W, Z0[s], XU[s], order, "l1-linf")
        for k in range(steps):
            np.testing.assert_allclose(lo[s, k], hulls[k].left_limit, rtol=common.GEN_RTOL, atol=1e-12)
            np.testing.assert_allclose(hi[s, k], hulls[k].right_limit, rtol=common.GEN_RTOL, atol=1e-12)
        np.testing.assert_allclose(Zf[s, :, 1:1 + gf[s]], Zo.generators, rtol=1e-8, atol=1e-12)


# ---- shapes refused before any launch --------------------------------------------------------------------------------
def _reach_ok(S=3, n=4, p=5, N=2, g=3, gW=1, per=False):
    lead = (S,) if per else ()
    return dict(Cm=torch.zeros(lead + (n, p)), Gm=torch.zeros(lead + (N, n, p)), Z=torch.zeros((S, p, 1 + g)),
                W=torch.zeros((n, 1 + gW)))


REACH_BAD = {
    "Cm-cols": ("Cm", lambda a: dict(a, Cm=torch.zeros(4, 6))),
    "Cm-per-S": ("Cm", lambda a: dict(a, Cm=torch.zeros(2, 4, 5), Gm=torch.zeros(2, 2, 4, 5))),
    "Cm-1d": ("Cm", lambda a: dict(a, Cm=torch.zeros(20))),
    "Gm-rows": ("Gm", lambda a: dict(a, Gm=torch.zeros(2, 3, 5))),
    "Gm-cols": ("Gm", lambda a: dict(a, Gm=torch.zeros(2, 4, 6))),
    "Gm-shared-with-per-Cm": ("Gm", lambda a: dict(a, Cm=torch.zeros(3, 4, 5))),
    "Gm-per-with-shared-Cm": ("Gm", lambda a: dict(a, Gm=torch.zeros(3, 2, 4, 5))),
    "Gm-per-S": ("Gm", lambda a: dict(a, Cm=torch.zeros(3, 4, 5), Gm=torch.zeros(2, 2, 4, 5))),
    "Z-2d": ("Z", lambda a: dict(a, Z=torch.zeros(5, 4))),
    "W-rows": ("W", lambda a: dict(a, W=torch.zeros(3, 2))),
    "W-no-centre": ("W", lambda a: dict(a, W=torch.zeros(4, 0))),
    "W-1d": ("W", lambda a: dict(a, W=torch.zeros(4))),
}


@pytest.mark.parametrize("name", list(REACH_BAD))
def test_reach_step_rejects_malformed_shapes(T, name):
    what, bad = REACH_BAD[name]
    a = {k: v.double().cuda() for k, v in bad(_reach_ok()).items()}
    torch.cuda.synchronize()
    with pytest.raises(AssertionError, match=rf"^{what}: "):
        T.ops.tzddpc.reach_step(a["Cm"], a["Gm"], a["Z"], a["W"])
    ok = {k: v.double().cuda() for k, v in _reach_ok().items()}
    assert T.ops.tzddpc.reach_step(ok["Cm"], ok["Gm"], ok["Z"], ok["W"]).shape == (3, 4, 3 * 4 + 1)


def _tube_ok(S=3, n=4, m=2, NK=2, ND=3, steps=2, gW=1, per=False):
    lead = (S,) if per else ()
    return dict(CK=torch.zeros(lead + (n, n)), GK=torch.zeros(lead + (NK, n, n)), GD=torch.zeros(lead + (ND, n, n + m)),
                Z0=torch.zeros((S, n, 2)), XU=torch.zeros((S, steps, n + m)), W=torch.zeros((n, 1 + gW)))


TUBE_BAD = {
    "CK-square": ("CK", lambda a: dict(a, CK=torch.zeros(4, 5))),
    "CK-per-S": ("CK", lambda a: dict(a, CK=torch.zeros(2, 4, 4), GK=torch.zeros(2, 2, 4, 4), GD=torch.zeros(2, 3, 4, 6))),
    "GK-shared-with-per-CK": ("GK", lambda a: dict(a, CK=torch.zeros(3, 4, 4))),
    "GK-per-with-shared-CK": ("GK", lambda a: dict(a, GK=torch.zeros(3, 2, 4, 4))),
    "GK-rows": ("GK", lambda a: dict(a, GK=torch.zeros(2, 3, 4))),
    "GK-per-S": ("GK", lambda a: dict(a, CK=torch.zeros(3, 4, 4), GK=torch.zeros(2, 2, 4, 4), GD=torch.zeros(3, 3, 4, 6))),
    "GD-shared-with-per-CK": ("GD", lambda a: dict(a, CK=torch.zeros(3, 4, 4), GK=torch.zeros(3, 2, 4, 4))),
    "GD-cols": ("GD", lambda a: dict(a, GD=torch.zeros(3, 4, 5))),
    "GD-rows": ("GD", lambda a: dict(a, GD=torch.zeros(3, 5, 6))),
    "GD-per-S": ("GD", lambda a: dict(a, CK=torch.zeros(3, 4, 4), GK=torch.zeros(3, 2, 4, 4), GD=torch.zeros(2, 3, 4, 6))),
    "Z0-2d": ("Z0", lambda a: dict(a, Z0=torch.zeros(4, 2))),
    "XU-S": ("XU", lambda a: dict(a, XU=torch.zeros(2, 2, 6))),
    "XU-no-input": ("XU", lambda a: dict(a, XU=torch.zeros(3, 2, 4), GD=torch.zeros(3, 4, 4))),
    "W-rows": ("W", lambda a: dict(a, W=torch.zeros(5, 2))),
    "W-no-centre": ("W", lambda a: dict(a, W=torch.zeros(4, 0))),
}


@pytest.mark.parametrize("name", list(TUBE_BAD))
def test_tube_rollout_rejects_malformed_shapes(T, name):
    what, bad = TUBE_BAD[name]
    a = {k: v.double().cuda() for k, v in bad(_tube_ok()).items()}
    torch.cuda.synchronize()
    with pytest.raises(AssertionError, match=rf"^{what}: "):
        T.ops.tzddpc.tube_rollout(a["CK"], a["GK"], a["GD"], a["Z0"], a["XU"], a["W"], 2.0, 0, 8)
    ok = {k: v.double().cuda() for k, v in _tube_ok().items()}
    Zf, gf, lo, hi = T.ops.tzddpc.tube_rollout(ok["CK"], ok["GK"], ok["GD"], ok["Z0"], ok["XU"], ok["W"], 2.0, 0, 8)
    assert Zf.shape == (3, 4, 9) and lo.shape == (3, 2, 4)
