"""Shared inputs of the dense-matrix tests: continuous dosages in [0, 2] with missing entries, and the fit cases."""
import numpy as np

from mendeliht_jl_b200 import synth
from oracle import snp

N, P, K = 1200, 2500, 5


def continuous_dosages(seed: int, n: int, p: int, missing_rate: float = 0.01, noise: float = 0.3) -> np.ndarray:
    """Imputed-dosage-like matrix: the integer genotypes of synth.packed_columns plus uniform noise, clipped to [0, 2],
    NaN where the genotype is missing (float64, C order)."""
    bed = synth.packed_columns(seed, n, np.arange(p), missing_rate)
    g = snp.dosages(bed, n)
    rng = np.random.default_rng(seed + 1)
    return np.clip(g + rng.uniform(-noise, noise, size=g.shape), 0.0, 2.0)


def case_data(seed: int, d: str, ncov: int, n: int = N, p: int = P, k: int = K):
    """(y, z, x_raw): the response simulated from the integer genotypes, the dosages they blur."""
    y, z, *_ = synth.simulate_response(seed, n, p, k, d, n_cov=ncov, missing_rate=0.01)
    return y, z, continuous_dosages(seed, n, p)


# (id, d, l, ncov, fit keywords)
FIT_CASES = [
    ("normal", "Normal", "IdentityLink", 2, {"k": 7}),
    ("bernoulli_zkeep", "Bernoulli", "LogitLink", 2, {"k": 6, "zkeep": [True, False, True]}),
    ("poisson_weights", "Poisson", "LogLink", 1, {"k": 6, "weight": "random"}),
    ("negbin", "NegativeBinomial", "LogLink", 0, {"k": 6, "nb_r": 10.0}),
    ("negbin_mm", "NegativeBinomial", "LogLink", 0, {"k": 6, "est_r": "MM", "nb_r": 1.0}),
    ("negbin_newton", "NegativeBinomial", "LogLink", 0, {"k": 6, "est_r": "Newton", "nb_r": 1.0}),
    ("normal_init_beta", "Normal", "IdentityLink", 1, {"k": 6, "init_beta": True}),
    ("bernoulli_debias", "Bernoulli", "LogitLink", 1, {"k": 5, "debias": True}),
    ("normal_groups", "Normal", "IdentityLink", 1, {"k": "groups", "J": 3}),
    ("bernoulli_probit", "Bernoulli", "ProbitLink", 1, {"k": 5}),
    ("bernoulli_cloglog", "Bernoulli", "CloglogLink", 1, {"k": 5}),
]


def fit_kwargs(kw: dict, p: int) -> dict:
    """Materialises the symbolic entries of a case: weight='random' -> seeded prior weights in [1, 3], k='groups' -> a
    per-group k vector over 5 contiguous blocks."""
    kw = dict(kw)
    if kw.get("weight") == "random":
        rng = np.random.default_rng(7)
        kw["weight"] = rng.uniform(1.0, 3.0, size=p)
    if kw.get("k") == "groups":
        kw["group"] = np.repeat(np.arange(1, 6), -(-p // 5))[:p]
        kw["k"] = np.array([2, 1, 2, 1, 2])
    return kw
