"""Pins the oracle's SnpLinAlg options (scale, impute) on a small hand-written genotype matrix, because the GPU tests of
handles built with those options (test_gpu_handle_options.py) are only as good as the oracle.  CPU only."""
import itertools
import math

import numpy as np
import pytest

from oracle import snp

# dosages, -1 = missing: a mixed column, one without missing entries, a monomorphic one (mu = 0, sinv = 1), one whose
# observed entries are all 2 (mu = 2, sinv = 1) and one that is mostly missing
G = np.array([[0, 1, 0, 2, -1],
              [1, 2, 0, 2, 2],
              [-1, 0, -1, -1, -1],
              [2, 1, 0, 2, -1],
              [1, 1, 0, -1, 1],
              [0, 2, 0, 2, -1],
              [-1, 0, 0, 2, -1],
              [2, 1, 0, 2, 0],
              [1, 0, 0, 2, -1]])


def _by_hand(scale, impute):
    """x_ij = ((missing ? (impute ? mu_j : 0) : g_ij) - mu_j) * sinv_j, mu_j the mean of the observed dosages,
    sinv_j = 1 / sqrt(mu_j (1 - mu_j / 2)) when scaled and that is finite, else 1 -- one column at a time"""
    n, p = G.shape
    x = np.empty((n, p))
    for j in range(p):
        obs = [int(g) for g in G[:, j] if g >= 0]
        mu = sum(obs) / len(obs)
        s = math.sqrt(mu * (1.0 - mu / 2.0))
        sinv = 1.0 / s if scale and s > 0 else 1.0
        for i in range(n):
            g = float(G[i, j]) if G[i, j] >= 0 else (mu if impute else 0.0)
            x[i, j] = (g - mu) * sinv
    return x


@pytest.mark.parametrize("scale,impute", list(itertools.product([True, False], repeat=2)))
def test_options_by_hand(scale, impute):
    n = G.shape[0]
    bed = snp.pack_codes(snp.dosage_to_codes(G))
    o = snp.SnpLinAlgOracle(bed, n, scale=scale, impute=impute)
    x = o.dense()
    # the same IEEE operations in the same order: equal bit for bit
    np.testing.assert_array_equal(x, _by_hand(scale, impute))
    assert np.array_equal(o.nmiss, (G < 0).sum(axis=0))
    if not scale:
        assert np.all(o.sigma_inv == 1.0)
    assert o.sigma_inv[2] == 1.0 and o.sigma_inv[3] == 1.0
    # a missing entry: 0 with impute; 0 - mu_j = -2 in the column whose observed entries are all 2 without
    assert x[2, 3] == (0.0 if impute else -2.0)
    assert x[2, 2] == 0.0                                   # mu = 0: missing is 0 either way
    rng = np.random.default_rng(7)
    V = rng.normal(size=(n, 3)) + np.array([5.0, -40.0, 0.0])
    for v in (V[:, 0], V):
        want = x.T @ v
        np.testing.assert_allclose(o.xt_v(v), want, rtol=0, atol=1e-12 * np.abs(want).max())
    if not impute:                                          # the options change X'v for a right-hand side of large mean
        dflt = snp.SnpLinAlgOracle(bed, n, scale=scale).xt_v(V[:, 0])
        assert np.max(np.abs(o.xt_v(V[:, 0]) - dflt)) > 1e-3 * np.abs(dflt).max()
