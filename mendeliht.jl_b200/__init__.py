"""mendeliht.jl_b200 — B200 (sm_100a) implementation of MendelIHT.jl's IHT hot path.

The directory name contains a dot, so import it as `mendeliht_jl_b200` (the loader module at the repo root).
Everything numerical happens in libihtb200.so (hand-written CUDA, C ABI in include/ihtb200.h); this package is the
host-side mirror of the reference's Julia API.  There is no CPU fallback.
"""
from . import _lib, bgen, synth
from ._lib import (SWEEP_EXACT, SWEEP_FAST, SWEEP_PAIR, CudaError, DimensionMismatch, IHTBError, NumericError, device_count,
                   launch_count, load)
from .api import (BERNOULLI, NEGBIN, NORMAL, POISSON, B200DenseLinAlg, B200MultiSnpLinAlg, B200SnpLinAlg, IHTResult, IHTVariable, mIHTResult, mIHTVariable,
                  is_multivariate, allocate_fold_and_k,
                  canonicallink, cross_validate, cv_iht, cv_run, fit_iht, iht, maf_weights, meanloss, parse_covariates)

__all__ = ["B200SnpLinAlg", "B200DenseLinAlg", "B200MultiSnpLinAlg", "IHTResult", "IHTVariable", "fit_iht", "cv_iht", "cv_run", "allocate_fold_and_k", "meanloss",
           "canonicallink", "maf_weights", "iht", "cross_validate", "parse_covariates", "NORMAL", "BERNOULLI", "POISSON", "NEGBIN", "SWEEP_FAST", "SWEEP_EXACT", "SWEEP_PAIR", "load",
           "device_count", "launch_count", "IHTBError", "DimensionMismatch", "NumericError", "CudaError", "synth", "bgen"]
