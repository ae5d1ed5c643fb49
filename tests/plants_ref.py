"""numpy restatements of the per-scenario plant paths of tzddpc_b200/csrc/tz_rng.cu (test infrastructure), on the random
stream of oracle/philox.py:

    sample_plants                 tz_sample_plants (Philox purpose 6)
    generate_trajectories_plants  tz_generate_trajectories_plants (oracle.philox.generate_trajectories with a plant per data set)
"""
from __future__ import annotations

import numpy as np

from oracle.philox import draws


def generate_trajectories_plants(A, B, X0Z, UZ, WZ, S: int, T: int, seed: int, scenario_offset: int = 0):
    """examples/utils.py:6-45 for S data sets, data set s from the plant (A[s], B[s]): A (S, n, n), B (S, n, m).
    Returns U (S, T, m), X (S, T, n)."""
    n, m = B.shape[-2:]
    sid = scenario_offset + np.arange(S)
    x = X0Z[:, 0][None] + draws(seed, sid, 0, 3, X0Z.shape[1] - 1, False) @ X0Z[:, 1:].T
    U = np.zeros((S, T, m))
    X = np.zeros((S, T, n))
    for t in range(T):
        u = UZ[:, 0][None] + draws(seed, sid, t, 1, UZ.shape[1] - 1, False) @ UZ[:, 1:].T
        U[:, t] = u
        if t + 1 < T:
            w = WZ[:, 0][None] + draws(seed, sid, t, 2, WZ.shape[1] - 1, True) @ WZ[:, 1:].T
            x = np.einsum("sij,sj->si", A, x) + np.einsum("sij,sj->si", B, u) + w
            X[:, t + 1] = x
    return U, X


def sample_plants(AB, Pinv, WZ, dataset, S: int, seed: int, scenario_offset: int = 0) -> np.ndarray:
    """tz_sample_plants: [A B] = AB_d - G_W R,  R[k, :] = sum_j beta_kj Pinv_d[j, :],  beta_kj = draw k (T-1) + j of
    (scenario_offset + s, t = 0, purpose 6) -- the point sum_g beta_g G_g of the generators G_g = -G_W[:, k] Pinv_d[j, :] of
    M_Sigma around its centre AB_d.  AB (D, n, n+m), Pinv (D, T-1, n+m), WZ (n, 1+gW), dataset (S,) or None (data set 0).
    Returns (S, n, n+m)."""
    AB, Pinv, WZ = (np.asarray(a, dtype=np.float64) for a in (AB, Pinv, WZ))
    d = np.zeros(S, dtype=np.int64) if dataset is None else np.asarray(dataset, dtype=np.int64)
    Tm, gW = Pinv.shape[1], WZ.shape[1] - 1
    beta = draws(seed, scenario_offset + np.arange(S), 0, 6, gW * Tm, False).reshape(S, gW, Tm)
    R = np.einsum("skj,sjc->skc", beta, Pinv[d])                  # (S, gW, n+m)
    return AB[d] - np.einsum("ik,skc->sic", WZ[:, 1:], R)
