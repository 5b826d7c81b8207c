"""Oracle (test infrastructure): dense design matrix, numpy restatement.

Restates what MendelIHT does with a dense `x::AbstractMatrix{T}` (reference `src/fit.jl:62`): `mul!(df, Transpose(x), r)`
is the plain product x' r, and `update_xb!` adds the columns of the support one after the other
(`src/utilities.jl:95-111`).  `standardize=True` restates `standardize_genotypes!` (`src/wrapper.jl:406-423`): NaN is
missing, mu_j is the mean of the observed entries, sigma_j = sqrt(mu_j (1 - mu_j / 2)), a missing entry becomes mu_j, and
x_ij = (g_ij - mu_j) * (1 / sigma_j) (1 / sigma_j = 1 when sigma_j = 0).  The reference divides by sigma_j instead of
multiplying by its inverse; the two differ by at most one ulp per entry, and multiplying reproduces the PLINK operator's
getindex (`SnpLinAlgOracle.dense`) bit for bit on integer dosages.

`dtype` is the element type the matrix is stored in: float32 storage rounds every (standardized) entry to float32 once,
after which everything is FP64, as on the device.
"""
from __future__ import annotations

import numpy as np


def standardize_genotypes(x: np.ndarray):
    """standardize_genotypes! in float64: returns (x_std, mu, sigma_inv, n_missing)."""
    g = np.asarray(x, dtype=np.float64)
    miss = np.isnan(g)
    nmiss = miss.sum(axis=0).astype(np.int64)
    nobs = (g.shape[0] - nmiss).astype(np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        mu = np.where(miss, 0.0, g).sum(axis=0) / nobs
    s = np.sqrt(mu * (1.0 - mu / 2.0))
    with np.errstate(divide="ignore", invalid="ignore"):
        sinv = np.where(s > 0, 1.0 / s, 1.0)
    xs = (np.where(miss, mu[None, :], g) - mu[None, :]) * sinv[None, :]
    return xs, mu, sinv, nmiss


class DenseLinAlgOracle:
    """Dense float64 stand-in for a `B200DenseLinAlg` (the methods `oracle.iht.fit_iht` and `oracle.cv.cv_iht` use)."""

    def __init__(self, x: np.ndarray, standardize: bool = False, dtype=np.float64):
        x = np.asarray(x)
        if standardize:
            xs, self.mu, self.sigma_inv, self.nmiss = standardize_genotypes(x)
        else:
            xs = np.asarray(x, dtype=np.float64)
            self.mu, self.sigma_inv = np.zeros(xs.shape[1]), np.ones(xs.shape[1])
            self.nmiss = np.zeros(xs.shape[1], dtype=np.int64)
        self._x = np.asfortranarray(xs.astype(dtype, copy=False).astype(np.float64, copy=False))
        self.n, self.p = self._x.shape

    @property
    def shape(self):
        return (self.n, self.p)

    def dense(self) -> np.ndarray:
        return self._x

    def columns(self, cols) -> np.ndarray:
        return self._x[:, np.asarray(cols, dtype=np.int64)]

    def xt_v(self, v: np.ndarray) -> np.ndarray:
        """mul!(out, Transpose(x), v): the plain product, v [n] or [n, m]."""
        return self._x.T @ v

    def support_xb(self, idx, coef) -> np.ndarray:
        """sum_{j in idx} x[:, j] * coef_j, added in the order given (update_xb!, src/utilities.jl:95-106)."""
        out = np.zeros(self.n)
        for j, cj in zip(idx, coef):
            out += self._x[:, j] * cj
        return out
