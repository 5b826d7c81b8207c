"""PLINK handles built with the reference's other SnpLinAlg options, scale=false and impute=false, against the CPU oracle
built with the same options, in every kernel that reads them: column statistics, decode, x[:, idx] * b, the X'V sweeps
(EXACT / FAST / PAIR, 2-bit and ternary tiles), the exact re-scoring gathers, init_beta, debiasing, CV and the
multivariate fit.  The other tests use the defaults (scale = impute = true) only.

With impute=false a missing genotype counts 0 (its standardized value is -mu_j sinv_j), and the sweeps and gathers
correct their centred sums by -vbar nmiss_j instead of the sum of the centred right-hand side over the missing samples.
That term scales with the mean vbar of the right-hand side, which a fit with an intercept drives towards zero.  So the
sweeps are tested directly with right-hand sides of large mean, on columns with 5 - 30 % missing entries, and every
comparison against the oracle first checks that the oracle of the default handle lies at least 100 tolerances away:
a kernel that took the default branch would fail."""
import os
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import mendeliht_jl_b200 as m
from mendeliht_jl_b200 import synth
from oracle import cv as ocv
from oracle import iht, mviht, snp
from parity_helpers import RTOL, compare_fit, compare_mv_fit

FLAGS = [(1, 0), (0, 1), (0, 0)]           # (scale, impute); (1, 1) is the default every other test uses
FLAG_IDS = ["impute0", "scale0", "scale0-impute0"]
MODES = [m.SWEEP_FAST, m.SWEEP_EXACT]


def _handle(bed, n, scale, impute, tern=None):
    """from_bed_columns with the options; tern = "1" / "0" forces the ternary copy of the tiles on / off"""
    if tern is None:
        return m.B200SnpLinAlg.from_bed_columns(bed, n, scale=bool(scale), impute=bool(impute))
    os.environ["IHTB_TERN"] = tern
    try:
        return m.B200SnpLinAlg.from_bed_columns(bed, n, scale=bool(scale), impute=bool(impute))
    finally:
        os.environ.pop("IHTB_TERN", None)


def _oracle(bed, n, scale=1, impute=1):
    return snp.SnpLinAlgOracle(bed, n, scale=bool(scale), impute=bool(impute))


def _check_sweep(got, want, base, bound, what):
    """|got - want| <= bound entry by entry, where the default handle's reference `base` is >= 100 bounds from `want`"""
    assert np.max(np.abs(want - base) / bound) >= 100, ("inputs do not tell the branches apart", what)
    assert np.all(np.abs(got - want) <= bound), what


def _check_fits_differ(ref, base, rtol=RTOL):
    """the oracle fit on the options under test is not the default handle's fit: its support or iteration count
    differs, or a coefficient lies more than 100 tolerances away"""
    if ref.iter != base.iter or not np.array_equal(np.asarray(ref.beta) != 0, np.asarray(base.beta) != 0):
        return
    a = np.concatenate([np.ravel(ref.beta), np.ravel(ref.c)])
    b = np.concatenate([np.ravel(base.beta), np.ravel(base.c)])
    assert np.any(np.abs(a - b) > 100 * (rtol * np.abs(b) + 1e-12)), "inputs do not tell the branches apart"


# ---- statistics, decode, support product: same formula, same order of additions as the oracle -> bit for bit --------
@pytest.mark.parametrize("scale,impute", FLAGS, ids=FLAG_IDS)
@pytest.mark.parametrize("n,p,miss", [(1000, 257, 0.05), (1003, 300, 0.1), (515, 64, 0.3), (7, 5, 0.2), (2049, 130, 0.05)])
def test_stats_decode_support_bit_exact(n, p, miss, scale, impute):
    bed = synth.packed_columns(11, n, np.arange(p), miss)
    g = _handle(bed, n, scale, impute)
    d = m.B200SnpLinAlg.from_bed_columns(bed, n)
    o = _oracle(bed, n, scale, impute)
    mu, sinv, nm = g.stats()
    mu0, sinv0, nm0 = d.stats()
    assert np.array_equal(mu, mu0) and np.array_equal(nm, nm0)
    assert np.array_equal(mu, o.mu) and np.array_equal(nm, o.nmiss) and nm.sum() > 0
    assert np.array_equal(sinv, o.sigma_inv)
    assert np.all(sinv == 1.0) if not scale else np.array_equal(sinv, sinv0)
    x = g.decode()
    assert np.array_equal(x, o.dense())
    assert not np.array_equal(x, d.decode())
    assert np.array_equal(g.decode(3, min(n, 40), 1, min(p, 9)), o.dense()[3:min(n, 40), 1:min(p, 9)])
    rng = np.random.default_rng(2)
    k = min(p, 37)
    idx = np.sort(rng.permutation(p)[:k])
    coef = rng.normal(size=k)
    assert np.array_equal(g.x_support(idx, coef), o.support_xb(idx, coef))
    C5 = rng.normal(size=(k, 5))
    got = g.x_support(idx, C5)
    for t in range(5):
        assert np.array_equal(got[:, t], o.support_xb(idx, C5[:, t])), t
    assert np.array_equal(g.counts(), d.counts())
    assert np.array_equal(g.maf(), d.maf())
    assert np.array_equal(g.packed(), bed) and np.array_equal(d.packed(), bed)
    g.close(); d.close()


# ---- X'V in every mode, from both tile copies -------------------------------------------------------------------------
@pytest.mark.parametrize("scale,impute", FLAGS, ids=FLAG_IDS)
@pytest.mark.parametrize("n,p,miss", [(1003, 513, 0.05), (640, 9, 0.1), (641, 130, 0.3), (3200, 257, 0.05), (50, 4, 0.3),
                                      (12801, 1030, 0.05), (12801, 2050, 0.1)])
def test_sweeps_against_oracle(n, p, miss, scale, impute):
    """EXACT within 1e-11 max|ref|; FAST within 2^-18 ||u||_1 sinv_j; PAIR within 3.1 2^-11 ||u||_2 sgn_j (the bounds the
    fits assume; u = v - mean(v)).  Right-hand sides: large mean with a genetic signal (the sums of a few columns, as in
    a residual), the same at magnitude 1e-3 (paired with the first in PAIR mode), and mean near zero (the odd one out of
    the PAIR pass, which takes the FAST path)."""
    bed = synth.packed_columns(6, n, np.arange(p), miss)
    o = _oracle(bed, n, scale, impute)
    rng = np.random.default_rng(1)
    Z = rng.normal(size=(n, 3))
    signal = np.nan_to_num(snp.dosages(bed[np.arange(0, p, max(1, p // 5))[:5]], n)).sum(axis=1)
    V = np.column_stack([Z[:, 0] + 5.0 + signal, 1e-3 * (Z[:, 1] + 5.0 + signal), Z[:, 2]])
    want = o.xt_v(V)
    base = _oracle(bed, n).xt_v(V)
    U = V - V.mean(axis=0)
    hs = {tern: _handle(bed, n, scale, impute, tern) for tern in ("1", "0")}
    assert hs["1"].sweep_stream_bytes()[1] and not hs["0"].sweep_stream_bytes()[1]
    for tern, g in hs.items():
        _, sinv, _ = g.stats()
        assert np.array_equal(sinv, o.sigma_inv)
        cnt = g.counts()
        sgn = sinv * np.maximum(np.sqrt(cnt[2] + 4.0 * cnt[3]), 1.0)
        ex3 = g.xt_v(V, m.SWEEP_EXACT)
        pair = g.xt_v(V, m.SWEEP_PAIR)
        for t in range(3):
            tiny = 1e-12 * np.abs(want[:, t]).max()
            tol = 1e-11 * np.abs(want[:, t]).max()
            _check_sweep(g.xt_v(V[:, t], m.SWEEP_EXACT), want[:, t], base[:, t], tol, ("EXACT", tern, t))
            _check_sweep(ex3[:, t], want[:, t], base[:, t], tol, ("EXACT x3", tern, t))
            fast = (2.0 ** -18) * np.abs(U[:, t]).sum() * sinv + tiny
            _check_sweep(g.xt_v(V[:, t], m.SWEEP_FAST), want[:, t], base[:, t], fast, ("FAST", tern, t))
            paired = 3.1 * 2.0 ** -11 * np.sqrt((U[:, t] ** 2).sum()) * sgn + tiny if t < 2 else fast
            _check_sweep(pair[:, t], want[:, t], base[:, t], paired, ("PAIR", tern, t))
    assert np.array_equal(hs["1"].xt_v(V, m.SWEEP_EXACT), hs["0"].xt_v(V, m.SWEEP_EXACT))
    for g in hs.values():
        g.close()


# ---- exact re-scoring: nibble-table kernel (one right-hand side) against the per-column kernel ------------------------
@pytest.mark.parametrize("scale,impute", FLAGS, ids=FLAG_IDS)
@pytest.mark.parametrize("n,p,miss,ncols", [(1003, 300, 0.05, 257), (5000, 64, 0.1, 64), (513, 40, 0.3, 9),
                                            (40000, 128, 0.05, 500)])
def test_nibble_gather_matches_per_column_kernel(n, p, miss, ncols, scale, impute):
    g = _handle(synth.packed_columns(77, n, np.arange(p), miss), n, scale, impute)
    _, err = g.gather_bench(ncols, 1)
    assert err <= 1e-13, err
    g.close()


# ---- fits against the oracle --------------------------------------------------------------------------------------------
FIT_CASES = [
    # d, link, n, p, true k, fitted k, covariates (None: z=None, the intercept alone), missing rate
    ("Normal", "IdentityLink", 1200, 3000, 8, 10, 2, 0.1),
    ("Bernoulli", "LogitLink", 2000, 2500, 5, 7, 1, 0.05),
    ("Poisson", "LogLink", 1500, 2500, 6, 8, None, 0.15),
]


def _fit_data(d, n, p, k, ncov, miss):
    seed = 300 + n + p
    y, z, *_ = synth.simulate_response(seed, n, p, k, d, n_cov=ncov or 0, missing_rate=miss)
    return y, (None if ncov is None else z), synth.packed_columns(seed, n, np.arange(p), miss)


@pytest.mark.parametrize("scale,impute", FLAGS, ids=FLAG_IDS)
@pytest.mark.parametrize("d,l,n,p,k,kfit,ncov,miss", FIT_CASES)
def test_fit_matches_oracle(d, l, n, p, k, kfit, ncov, miss, scale, impute):
    y, z, bed = _fit_data(d, n, p, k, ncov, miss)
    g = _handle(bed, n, scale, impute)
    ref = iht.fit_iht(y, _oracle(bed, n, scale, impute), z, k=kfit, d=d, l=l)
    assert ref.iter < 200
    _check_fits_differ(ref, iht.fit_iht(y, _oracle(bed, n), z, k=kfit, d=d, l=l))
    for mode in MODES:
        compare_fit(m.fit_iht(y, g, z, k=kfit, d=d, l=l, sweep_mode=mode), ref)
    g.close()


OPTION_CASES = [
    # option, d, link, n, p, true k, fitted k, covariates, missing rate
    ("init_beta", "Normal", "IdentityLink", 1200, 2500, 6, 7, 2, 0.1),      # class sums, am = a0 for a missing entry
    ("debias", "Bernoulli", "LogitLink", 2000, 3000, 5, 7, 1, 0.05),        # IRLS refit on decoded support columns
    ("weight", "Poisson", "LogLink", 1500, 2500, 6, 8, 1, 0.1),
    ("group", "Normal", "IdentityLink", 1500, 3000, 6, 2, 1, 0.1),
]


def _option(name, g):
    if name == "init_beta":
        return {"init_beta": True}
    if name == "debias":
        return {"debias": True}
    if name == "weight":
        return {"weight": m.maf_weights(g, max_weight=5.0)}
    return {"J": 4, "group": np.arange(g.p) // 100 + 1}


@pytest.mark.parametrize("scale,impute", FLAGS, ids=FLAG_IDS)
@pytest.mark.parametrize("opt,d,l,n,p,k,kfit,ncov,miss", OPTION_CASES)
def test_fit_options_match_oracle(opt, d, l, n, p, k, kfit, ncov, miss, scale, impute):
    y, z, bed = _fit_data(d, n, p, k, ncov, miss)
    g = _handle(bed, n, scale, impute)
    kw = _option(opt, g)
    o = _oracle(bed, n, scale, impute)
    ref = iht.fit_iht(y, o, z, k=kfit, d=d, l=l, **kw)
    assert ref.iter < 200
    _check_fits_differ(ref, iht.fit_iht(y, _oracle(bed, n), z, k=kfit, d=d, l=l, **kw))
    plain = iht.fit_iht(y, o, z, k=kfit, d=d, l=l)
    assert ref.iter != plain.iter or not np.array_equal(ref.beta, plain.beta)      # the option is in effect here
    for mode in MODES:
        compare_fit(m.fit_iht(y, g, z, k=kfit, d=d, l=l, sweep_mode=mode, **kw), ref)
    g.close()


@pytest.mark.parametrize("scale,impute", FLAGS, ids=FLAG_IDS)
def test_cv_run_matches_oracle(scale, impute):
    """The whole grid in one call, with two fits at a time sharing a PAIR sweep (the default at this n), and one fit at a
    time: both equal the oracle's grid."""
    n, p, q, path = 1000, 2000, 3, [1, 3, 5, 8]
    y, z, bed = _fit_data("Poisson", n, p, 4, 1, 0.1)
    folds = synth.folds_for(21, n, q)
    g = _handle(bed, n, scale, impute)
    _, rgrid, riters = ocv.cv_iht(y, _oracle(bed, n, scale, impute), z, d="Poisson", l="LogLink", path=path, q=q,
                                  folds=folds, return_grid=True)
    _, bgrid, biters = ocv.cv_iht(y, _oracle(bed, n), z, d="Poisson", l="LogLink", path=path, q=q, folds=folds,
                                  return_grid=True)
    assert not np.array_equal(riters, biters) or np.max(np.abs(rgrid - bgrid) / bgrid) > 100 * RTOL
    assert riters.max() < 100
    mses, iters = m.cv_run(y, g, z, folds, q, path, d="Poisson", l="LogLink")
    os.environ["IHTB_CV_PAIR"] = "0"
    try:
        solo, solo_iters = m.cv_run(y, g, z, folds, q, path, d="Poisson", l="LogLink")
    finally:
        os.environ.pop("IHTB_CV_PAIR", None)
    assert np.array_equal(iters, riters) and np.array_equal(solo_iters, riters)
    np.testing.assert_allclose(mses, rgrid, rtol=RTOL)
    np.testing.assert_allclose(mses, solo, rtol=1e-10, atol=0)
    g.close()


def _mv_data(seed, n, p, r, k, miss):
    rng = np.random.default_rng(seed)
    bed = synth.packed_columns(seed, n, np.arange(p), miss)
    idx = np.sort(rng.permutation(p)[:k])
    B = np.zeros((r, k))
    for c in range(k):
        B[rng.integers(0, r), c] = rng.normal() * 0.8
    A = rng.normal(size=(r, r))
    E = np.linalg.cholesky(A @ A.T / r + np.eye(r) * 0.5) @ rng.normal(size=(r, n))
    Z = np.vstack([np.ones(n), rng.normal(size=n)])
    Y = B @ synth.standardized_columns(seed, n, idx, miss).T + rng.normal(size=(r, 2)) * 0.5 @ Z + E
    return bed, Y, Z


@pytest.mark.parametrize("scale,impute", FLAGS, ids=FLAG_IDS)
def test_mv_fit_matches_oracle(scale, impute):
    """MvNormal with r = 3 traits: the per-column gather with M = 3 right-hand sides, PAIR sweeps, multivariate init_beta."""
    n, p, r, k = 1500, 2000, 3, 9
    bed, Y, Z = _mv_data(45, n, p, r, k, 0.1)
    g = _handle(bed, n, scale, impute)
    o, o0 = _oracle(bed, n, scale, impute), _oracle(bed, n)
    for init in (False, True):
        ref = mviht.fit_mv_iht(Y, o, Z, k=k + 2, init_beta=init)
        _check_fits_differ(ref, mviht.fit_mv_iht(Y, o0, Z, k=k + 2, init_beta=init))
        for mode in ([m.SWEEP_FAST, m.SWEEP_PAIR] if not init else [m.SWEEP_FAST]):
            compare_mv_fit(m.fit_iht(Y, g, Z, k=k + 2, init_beta=init, sweep_mode=mode), ref)
    g.close()


# ---- ingest paths and sharding ------------------------------------------------------------------------------------------
def test_piecewise_ingest_carries_the_options(tmp_path):
    """from_bed_files (create_empty + load_columns + finalize) over three files == from_bed_columns, options included."""
    n, p, miss = 1003, 777, 0.1
    bed = synth.packed_columns(5, n, np.arange(p), miss)
    paths = []
    for a, b in [(0, 300), (300, 301), (301, p)]:
        path = tmp_path / f"chr{a}.bed"
        snp.write_bed(str(path), bed[a:b])
        paths.append(str(path))
    g = m.B200SnpLinAlg.from_bed_columns(bed, n, scale=False, impute=False)
    g2 = m.B200SnpLinAlg.from_bed_files(paths, n, scale=False, impute=False)
    assert np.array_equal(g2.packed(), g.packed())
    for a, b in zip(g2.stats(), g.stats()):
        assert np.array_equal(a, b)
    v = np.random.default_rng(0).normal(size=n) + 5.0
    got = g2.xt_v(v, m.SWEEP_EXACT)
    assert np.array_equal(got, g.xt_v(v, m.SWEEP_EXACT))
    want = _oracle(bed, n, 0, 0).xt_v(v)
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-11 * np.abs(want).max())
    g.close(); g2.close()


@pytest.mark.multigpu
def test_sharded_fit_with_options_matches_single_gpu():
    """A SHARD multi-device handle built with scale=false, impute=false reproduces the single-GPU fit on the same options
    (tolerances of test_gpu_multi: the all-reduce adds the shard partials in rank order)."""
    ngpu = min(m.device_count(), 8)
    n, p, k = 4000, 12000, 6
    y, z, *_ = synth.simulate_response(57, n, p, k, "Normal", n_cov=1, missing_rate=0.1)
    bed = synth.packed_columns(57, n, np.arange(p), 0.1)
    gm = m.B200MultiSnpLinAlg.from_bed_columns(bed, n, ngpu=ngpu, mode=m.B200MultiSnpLinAlg.SHARD, scale=False,
                                               impute=False)
    g1 = m.B200SnpLinAlg.from_bed_columns(bed, n, scale=False, impute=False)
    for kw in ({"sweep_mode": m.SWEEP_FAST}, {"sweep_mode": m.SWEEP_EXACT}, {"init_beta": True}):
        res = m.fit_iht(y, gm, z, k=k + 2, **kw)
        ref = m.fit_iht(y, g1, z, k=k + 2, **kw)
        assert res.iter == ref.iter and np.array_equal(np.flatnonzero(res.beta), np.flatnonzero(ref.beta))
        assert [t[1] for t in res.trace] == [t[1] for t in ref.trace]
        np.testing.assert_allclose(res.beta, ref.beta, rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(res.c, ref.c, rtol=1e-9, atol=1e-12)
        assert abs(res.logl - ref.logl) <= 1e-9 * abs(ref.logl)
    gm.close(); g1.close()


# ---- center=false is rejected, as by the reference ----------------------------------------------------------------------
def test_uncentered_handles_are_rejected(tmp_path):
    n, p = 100, 12
    bed = synth.packed_columns(3, n, np.arange(p), 0.1)
    path = tmp_path / "x.bed"
    snp.write_bed(str(path), bed)
    msg = re.escape("x is not centered! Please construct SnpLinAlg{Float64}(::SnpArray, center=true, scale=true)")
    for make in (lambda: m.B200SnpLinAlg.from_bed_columns(bed, n, center=False),
                 lambda: m.B200SnpLinAlg.from_bed_columns(bed, n, center=False, scale=False, impute=False),
                 lambda: m.B200SnpLinAlg.from_bed_files([str(path)], n, center=False),
                 lambda: m.B200MultiSnpLinAlg.from_bed_columns(bed, n, ngpu=1, center=False)):
        with pytest.raises(m.IHTBError, match=msg) as e:
            make()
        assert e.value.code == m._lib.IHTB_EUNSUPPORTED
