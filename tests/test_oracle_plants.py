"""The numpy restatements of the per-scenario plant paths (tests/plants_ref.py), without a GPU: sample_plants against the
explicit generators of M_Sigma = (X1 - M_w) pinv([X0; U0]) built by oracle/zono.py, and the per-data-set trajectory
generator against the shared one."""
import numpy as np

from oracle import philox
from oracle.zono import Zonotope, compute_LTI_matrix_zonotope, concatenate_zonotope
from tests import plants_ref


def _data(seed, T=12, n=3, m=2):
    rng = np.random.default_rng(seed)
    A = 0.5 * rng.standard_normal((n, n))
    B = rng.standard_normal((n, m))
    W = Zonotope(np.array([0.01, -0.02, 0.0][:n]), 0.05 * rng.standard_normal((n, 2)))
    X0Z = np.hstack([np.zeros((n, 1)), np.eye(n)])
    UZ = np.hstack([np.zeros((m, 1)), np.eye(m)])
    U, X = philox.generate_trajectories(A, B, X0Z, UZ, _wz(W), 1, T, seed)
    return W, U[0], X[0]


def _wz(W):
    return np.hstack([W.center[:, None], W.generators])


def test_sample_plants_is_a_point_of_the_explicit_msigma():
    for seed in (1, 2):
        W, U, X = _data(seed)
        T = X.shape[0]
        Mw = concatenate_zonotope(W, T - 1)
        M = compute_LTI_matrix_zonotope(X[:-1], X[1:], U[:-1], Mw)
        G = np.asarray(M.generators)                      # (gW (T-1), n, n+m), generator g = k (T-1) + j
        assert G.shape[0] == W.num_generators * (T - 1)
        Pinv = np.linalg.pinv(np.vstack([X[:-1].T, U[:-1].T]))
        S, off = 37, 1000
        got = plants_ref.sample_plants(np.asarray(M.center)[None], Pinv[None], _wz(W), None, S, seed=9, scenario_offset=off)
        beta = philox.draws(9, off + np.arange(S), 0, 6, G.shape[0], False)
        want = np.asarray(M.center)[None] + np.einsum("sg,gij->sij", beta, G)
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-12)
        # every sample lies in M_Sigma, the box of its generators
        assert all(M.contains(p) for p in got[:5])


def test_sample_plants_dataset_map_and_offsets():
    Ws, ABs, Ps = [], [], []
    for seed in (3, 4, 5):
        W, U, X = _data(seed)
        Ws.append(W)
        Pinv = np.linalg.pinv(np.vstack([X[:-1].T, U[:-1].T]))
        ABs.append((X[1:].T - W.center[:, None]) @ Pinv)
        Ps.append(Pinv)
    WZ = _wz(Ws[0])
    AB, P = np.stack(ABs), np.stack(Ps)
    ds = np.array([2, 0, 1, 1, 2, 0, 0, 2])
    full = plants_ref.sample_plants(AB, P, WZ, ds, len(ds), seed=4, scenario_offset=0)
    for s, d in enumerate(ds):
        one = plants_ref.sample_plants(AB[d:d + 1], P[d:d + 1], WZ, None, 1, seed=4, scenario_offset=s)
        np.testing.assert_array_equal(full[s], one[0])
    # a split batch draws the same plants
    np.testing.assert_array_equal(np.concatenate([plants_ref.sample_plants(AB, P, WZ, ds[:3], 3, 4, 0),
                                                  plants_ref.sample_plants(AB, P, WZ, ds[3:], 5, 4, 3)]), full)


def test_generate_trajectories_plants_equals_the_shared_call_per_plant():
    rng = np.random.default_rng(7)
    n, m, S, T = 2, 1, 5, 9
    A = np.array([[1.0, 0.1], [0.0, 1.0]]) * (1 + 0.02 * rng.uniform(-1, 1, (S, 1, 1)))
    B = np.array([[0.0], [0.1]]) * (1 + 0.02 * rng.uniform(-1, 1, (S, 1, 1)))
    X0Z = np.array([[0.0, 1.0, 0.0], [0.0, 0.0, 1.0]])
    UZ = np.array([[0.0, 1.0]])
    WZ = np.array([[0.0, 0.01, 0.0], [0.0, 0.0, 0.01]])
    U, X = plants_ref.generate_trajectories_plants(A, B, X0Z, UZ, WZ, S, T, seed=3)
    for s in range(S):
        Us, Xs = philox.generate_trajectories(A[s], B[s], X0Z, UZ, WZ, 1, T, seed=3, scenario_offset=s)
        np.testing.assert_allclose(U[s], Us[0], rtol=0, atol=1e-15)
        np.testing.assert_allclose(X[s], Xs[0], rtol=1e-13, atol=1e-15)
