"""16-bit fixed-point dosages (B200DenseLinAlg.from_dosages, ihtb_geno_create_dosage16) on the GPU: exhaustive decode,
bit-for-bit equality with the Float64 handle of the same values (decode, stats, support matvec, fits, CV), D = 1 against
the PLINK handle, the X'v sweep against numpy and against its documented error bound, determinism, piecewise loading
and the rejected cases."""
import ctypes as C
import math
from fractions import Fraction

import numpy as np
import pytest

import mendeliht_jl_b200 as m
from mendeliht_jl_b200 import _lib, synth
from oracle import cv as ocv
from oracle import iht, snp
from oracle.dense import DenseLinAlgOracle
from parity_helpers import compare_fit
from dense_cases import FIT_CASES, P, case_data, continuous_dosages, fit_kwargs

pytestmark = pytest.mark.gpu

F16 = m.B200DenseLinAlg.from_dosages
F64 = m.B200DenseLinAlg.from_array


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _same_bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape and np.array_equal(_bits(a), _bits(b))


def _grid_values(seed, n, p, den, miss=0.0, extra_ld=0):
    """[n, p] float64 dosages on the grid 1/den in [0, 2] (a view with leading dimension n + extra_ld), NaN at `miss`"""
    rng = np.random.default_rng(seed)
    big = np.asfortranarray(np.rint(rng.uniform(0.0, 2.0, size=(n + extra_ld, p)) * den) / den)
    if miss:
        big[rng.random(big.shape) < miss] = np.nan
    return big[:n]


def _quantised(x_raw, den):
    return np.rint(x_raw * den) / den                      # NaN stays NaN


@pytest.mark.parametrize("den", [1, 3, 255, 1000, 16384, 32767])
def test_decode_every_code(den):
    n = 4099
    codes = np.zeros(n * 16, dtype=np.uint16)
    codes[:65535] = np.arange(65535, dtype=np.uint16)
    codes = codes.reshape(16, n).T                         # [n, 16], column-major walk over 0..65534
    x = codes.astype(np.float64) / den
    d = F16(x, den)
    assert d.dtype == np.uint16 and d.denominator == den
    _same_bits(d.decode(), x)
    assert d.sweep_stream_bytes() == (2 * n * 16, False)
    mu, sinv, nm = d.stats()
    assert np.all(mu == 0) and np.all(sinv == 1) and np.all(nm == 0)


@pytest.mark.parametrize("standardize", [False, True])
@pytest.mark.parametrize("n,p,extra_ld", [(20, 517, 0), (1037, 333, 0), (4099, 130, 13)])
def test_equals_float64_handle(n, p, extra_ld, standardize):
    den = 16384
    x = _grid_values(n + p, n, p, den, miss=0.03 if standardize else 0.0, extra_ld=extra_ld)
    a, b = F16(x, den, standardize=standardize), F64(x, standardize=standardize)
    _same_bits(a.decode(), b.decode())
    _same_bits(a.decode(3, n - 1, 5, p - 2), b.decode(3, n - 1, 5, p - 2))
    (mu_a, si_a, nm_a), (mu_b, si_b, nm_b) = a.stats(), b.stats()
    _same_bits(mu_a, mu_b)
    _same_bits(si_a, si_b)
    assert np.array_equal(nm_a, nm_b)
    rng = np.random.default_rng(n)
    idx = rng.choice(p, size=min(p, 17), replace=False)
    coef = rng.standard_normal(idx.shape[0])
    _same_bits(a.x_support(idx, coef), b.x_support(idx, coef))
    C2 = rng.standard_normal((idx.shape[0], 2))
    _same_bits(a.x_support(idx, C2), b.x_support(idx, C2))
    # the C entry point with a host leading dimension > n reads the same handle
    codes = np.zeros((n + 7, p), dtype=np.uint16, order="F")
    codes[:n] = m.B200DenseLinAlg.encode_dosages(x, den, standardize)
    h = C.c_void_p()
    _lib.check(m.load().ihtb_geno_create_dosage16(codes.ctypes.data_as(C.POINTER(C.c_uint16)), n, p, n + 7, den,
                                                  int(standardize), C.byref(h)))
    c = m.B200DenseLinAlg(h, n, p, np.uint16, standardize, den)
    _same_bits(c.decode(), b.decode())


def test_integer_genotypes_equal_plink_handle(normal_data):
    n, bed, y, z = normal_data["n"], normal_data["bed"], normal_data["y"], normal_data["z"]
    g = m.B200SnpLinAlg.from_bed_columns(bed, n)
    d = F16(snp.dosages(bed, n), 1, standardize=True)
    _same_bits(d.decode(), g.decode())
    a = m.fit_iht(y, g, z, k=7, d="Normal", l="IdentityLink")
    b = m.fit_iht(y, d, z, k=7, d="Normal", l="IdentityLink")
    assert a.iter == b.iter and [t[1] for t in a.trace] == [t[1] for t in b.trace]
    assert np.array_equal(np.flatnonzero(a.beta), np.flatnonzero(b.beta))
    np.testing.assert_allclose(b.beta, a.beta, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(b.c, a.c, rtol=1e-9, atol=1e-12)
    assert abs(a.logl - b.logl) <= 1e-9 * abs(a.logl)


def test_integer_genotypes_with_missing_equal_plink_handle():
    n, p = 1500, 3000
    y, z, *_ = synth.simulate_response(77, n, p, 5, "Bernoulli", n_cov=1, missing_rate=0.02)
    bed = synth.packed_columns(77, n, np.arange(p), 0.02)
    g = m.B200SnpLinAlg.from_bed_columns(bed, n)
    d = F16(snp.dosages(bed, n), 1, standardize=True)
    _same_bits(d.decode(), g.decode())
    a = m.fit_iht(y, g, z, k=5, d="Bernoulli", l="LogitLink")
    b = m.fit_iht(y, d, z, k=5, d="Bernoulli", l="LogitLink")
    assert a.iter == b.iter and np.array_equal(np.flatnonzero(a.beta), np.flatnonzero(b.beta))
    np.testing.assert_allclose(b.beta, a.beta, rtol=1e-9, atol=1e-12)


@pytest.mark.parametrize("standardize", [False, True])
@pytest.mark.parametrize("n,p,extra_ld", [(20, 517, 0), (1037, 333, 0), (4099, 130, 13)])
def test_xt_v_matches_numpy(n, p, extra_ld, standardize):
    x = _grid_values(7 * n + p, n, p, 1000, miss=0.03 if standardize else 0.0, extra_ld=extra_ld)
    d = F16(x, 1000, standardize=standardize)
    xd = d.decode()
    rng = np.random.default_rng(p)
    for mm in (1, 3, 6):
        V = rng.standard_normal((n, mm)) + 0.7
        ref = xd.T @ V
        for mode in (m.SWEEP_FAST, m.SWEEP_EXACT):
            out = d.xt_v(V, mode)
            np.testing.assert_allclose(out, ref, rtol=1e-12, atol=1e-12 * np.abs(ref).max())
    v = rng.standard_normal(n) + 2.0
    np.testing.assert_allclose(d.xt_v(v), xd.T @ v, rtol=1e-12, atol=1e-12 * np.abs(xd.T @ v).max())


def _fix16_bound_coef(n, max_nmiss):
    """fix16_bound_coef (dense.cu): 2 (N_s + N_v + N_m + N_r + 9) 2^-53"""
    ld = -(-n // 256) * 256
    slabs, splits = -(-ld // 2048), -(-n // 8192)
    ns, nv, nr = 64 + 5 + slabs, 8 + 10 + slabs, 32 + 10 + splits
    return 2.0 * (ns + nv + max_nmiss + nr + 9) * 2.0 ** -53


def test_xt_v_within_documented_bound():
    n, den = 2300, 16384
    rng = np.random.default_rng(5)
    cols = []
    c = np.zeros(n); c[rng.choice(n, 3, replace=False)] = 1.0 / den; cols.append(c)          # mu ~ 1e-7: sinv ~ 4e3
    c = np.full(n, 2.0); c[rng.choice(n, 5, replace=False)] = 2.0 - 3.0 / den; cols.append(c)   # mu ~ 2
    c = np.rint(rng.uniform(0, 2, n) * den) / den; c[rng.random(n) < 0.5] = np.nan; cols.append(c)   # half missing
    c = np.rint(rng.uniform(0, 2, n) * den) / den; cols.append(c)                             # generic
    x = np.stack(cols, axis=1)
    d = F16(x, den, standardize=True)
    mu, sinv, nm = d.stats()
    xh = d.decode()
    g = np.where(np.isnan(x), -np.inf, x)
    scale = sinv * (g.max(axis=0) + np.abs(mu)) + np.abs(xh).max(axis=0)
    coef = _fix16_bound_coef(n, int(nm.max()))
    for v in (rng.standard_normal(n) + 1e6, rng.standard_normal(n), rng.uniform(-1, 1, n) * 1e-3 + 0.5):
        out = d.xt_v(v, m.SWEEP_FAST)
        L = np.abs(v).sum() + abs(v.sum())
        vf = [Fraction(float(t)) for t in v]
        for j in range(x.shape[1]):
            exact = sum((Fraction(float(a)) * b for a, b in zip(xh[:, j], vf)), Fraction(0))
            err = abs(Fraction(float(out[j])) - exact)
            assert err <= Fraction(coef * scale[j] * L), (j, float(err), coef * scale[j] * L)


def _f16_f64_pair(x_raw, den):
    xq = _quantised(x_raw, den)
    return F16(xq, den, standardize=True), F64(xq, standardize=True), xq


def _assert_fits_equal(a, b, debias=False):
    assert a.iter == b.iter
    assert np.array_equal(np.flatnonzero(a.beta), np.flatnonzero(b.beta))
    assert [t[:4] for t in a.trace] == [t[:4] for t in b.trace]        # all but the candidate count
    if debias:
        np.testing.assert_allclose(a.beta, b.beta, rtol=1e-12, atol=0)
        np.testing.assert_allclose(a.c, b.c, rtol=1e-12, atol=1e-300)
    else:
        _same_bits(a.beta, b.beta)
        _same_bits(a.c, b.c)
        _same_bits(a.logl, b.logl)
        _same_bits(a.sigma_g, b.sigma_g)


@pytest.mark.parametrize("den", [1000, 16384])
@pytest.mark.parametrize("cid,d,l,ncov,kw", FIT_CASES, ids=[c[0] for c in FIT_CASES])
def test_fit_equals_float64_handle(cid, d, l, ncov, kw, den):
    seed = 300 + [c[0] for c in FIT_CASES].index(cid)
    y, z, x_raw = case_data(seed, d, ncov)
    a16, a64, xq = _f16_f64_pair(x_raw, den)
    kk = fit_kwargs(kw, P)
    res = m.fit_iht(y, a16, z, d=d, l=l, **kk)
    ref64 = m.fit_iht(y, a64, z, d=d, l=l, **kk)
    _assert_fits_equal(res, ref64, debias=bool(kk.get("debias")))
    ref = iht.fit_iht(y, DenseLinAlgOracle(xq, standardize=True), z, d=d, l=l, **kk)
    assert ref.iter < 200
    compare_fit(res, ref, rtol=1e-5 if kk.get("est_r", "None") != "None" or l not in
                ("IdentityLink", "LogitLink", "LogLink") else 1e-6)


def test_cv_equals_float64_handle():
    y, z, x_raw = case_data(401, "Poisson", 1)
    a16, a64, xq = _f16_f64_pair(x_raw, 1000)
    folds = synth.folds_for(23, y.shape[0], 3)
    path = [2, 5, 8]
    m16, i16 = m.cv_iht(y, a16, z, d="Poisson", l="LogLink", path=path, q=3, folds=folds, return_grid=True)
    m64, i64 = m.cv_iht(y, a64, z, d="Poisson", l="LogLink", path=path, q=3, folds=folds, return_grid=True)
    _same_bits(m16, m64)
    assert np.array_equal(i16, i64)
    r16, ri16 = m.cv_run(y, a16, z, folds, 3, path, d="Poisson", l="LogLink")
    r64, ri64 = m.cv_run(y, a64, z, folds, 3, path, d="Poisson", l="LogLink")
    _same_bits(r16, r64)
    assert np.array_equal(ri16, ri64)
    _, rgrid, riters = ocv.cv_iht(y, DenseLinAlgOracle(xq, standardize=True), z, d="Poisson", l="LogLink", path=path,
                                  q=3, folds=folds, return_grid=True)
    assert np.array_equal(i16, riters)
    np.testing.assert_allclose(m16, rgrid, rtol=1e-6)


def test_fit_is_deterministic():
    y, z, x_raw = case_data(301, "Bernoulli", 2)
    a16, _, _ = _f16_f64_pair(x_raw, 16384)
    a = m.fit_iht(y, a16, z, k=6, d="Bernoulli", l="LogitLink")
    b = m.fit_iht(y, a16, z, k=6, d="Bernoulli", l="LogitLink")
    assert a.beta.tobytes() == b.beta.tobytes() and a.c.tobytes() == b.c.tobytes() and a.trace == b.trace


def test_piecewise_load_out_of_order():
    n, p, den = 1037, 300, 255
    x = _grid_values(9, n, p, den, miss=0.03)
    codes = np.asfortranarray(m.B200DenseLinAlg.encode_dosages(x, den, True))
    lib = m.load()
    h = C.c_void_p()
    _lib.check(lib.ihtb_geno_create_dosage16_empty(n, p, den, 1, C.byref(h)))
    d = m.B200DenseLinAlg(h, n, p, np.uint16, True, den)
    for j0, j1 in ((200, 300), (0, 77), (77, 200)):
        blk = np.asfortranarray(codes[:, j0:j1])
        _lib.check(lib.ihtb_geno_load_dense_columns(h, C.c_void_p(blk.ctypes.data), n, j0, j1 - j0))
    _lib.check(lib.ihtb_geno_finalize(h))
    ref = F16(x, den, standardize=True)
    _same_bits(d.decode(), ref.decode())
    for u, v in zip(d.stats(), ref.stats()):
        assert np.array_equal(u, v, equal_nan=True)
    v = np.random.default_rng(1).standard_normal(n)
    _same_bits(d.xt_v(v), ref.xt_v(v))


def test_rejected_cases():
    n, p = 300, 50
    x = _quantised(continuous_dosages(5, n, p), 1000)
    d = F16(x, 1000, standardize=True)
    lib = m.load()
    buf = np.zeros(4 * p, dtype=np.int64)
    assert lib.ihtb_geno_counts(d._h, _lib.ptr(buf, C.c_int64)) == _lib.IHTB_EUNSUPPORTED
    assert lib.ihtb_geno_maf(d._h, _lib.ptr(np.zeros(p), C.c_double)) == _lib.IHTB_EUNSUPPORTED
    assert lib.ihtb_geno_packed(d._h, 0, 1, _lib.ptr(np.zeros(n, np.uint8), C.c_uint8)) == _lib.IHTB_EUNSUPPORTED
    assert lib.ihtb_geno_ternary_tiles(d._h, _lib.ptr(np.zeros(8, np.uint8), C.c_uint8), 8) == _lib.IHTB_EUNSUPPORTED
    ms, err = C.c_double(), C.c_double()
    assert lib.ihtb_gather_bench(d._h, 4, 1, C.byref(ms), C.byref(err)) == _lib.IHTB_EUNSUPPORTED
    assert lib.ihtb_geno_set_offset(d._h, 3) == _lib.IHTB_EUNSUPPORTED
    assert lib.ihtb_geno_load_columns(d._h, _lib.ptr(np.zeros(8, np.uint8), C.c_uint8), 80, 0, 0) == _lib.IHTB_EINVAL
    codes = np.zeros((n, 1), dtype=np.uint16, order="F")
    assert lib.ihtb_geno_load_dense_columns(d._h, C.c_void_p(codes.ctypes.data), n, 0, 1) == _lib.IHTB_EINVAL  # ready
    Y = np.random.default_rng(1).standard_normal((2, n))
    with pytest.raises(m.IHTBError) as e:
        m.fit_iht(Y, d, np.ones((1, n)), k=3)
    assert e.value.code == _lib.IHTB_EUNSUPPORTED
    cfg = _lib.Cfg(0, 0, 3, 1.0, 1e-4, 10, 5, 3, 0, 0, 0)
    h = C.c_void_p()
    Yc = np.asfortranarray(Y.T)
    assert lib.ihtb_mvfit_create(d._h, Yc.ctypes.data_as(C.POINTER(C.c_double)), 2,
                                 _lib.ptr(np.ones(n), C.c_double), 1, C.byref(cfg), C.byref(h)) == _lib.IHTB_EUNSUPPORTED
    with pytest.raises(TypeError):
        m.maf_weights(d)
    xp = C.c_void_p(codes.ctypes.data)
    assert lib.ihtb_geno_create_dense(xp, _lib.DENSE_FIX16, n, 1, n, 0, C.byref(h)) == _lib.IHTB_EINVAL
    # the missing code without standardization: IHTB_EDOMAIN at finalize, as NaN is for float storage
    codes[3, 0] = _lib.DOSAGE16_MISSING
    assert lib.ihtb_geno_create_dosage16(codes.ctypes.data_as(C.POINTER(C.c_uint16)), n, 1, n, 1000, 0,
                                         C.byref(h)) == _lib.IHTB_EDOMAIN
    assert not h.value
    assert lib.ihtb_geno_create_dosage16(codes.ctypes.data_as(C.POINTER(C.c_uint16)), n, 1, n, 1000, 1,
                                         C.byref(h)) == _lib.IHTB_OK
    e = m.B200DenseLinAlg(h, n, 1, np.uint16, True, 1000)
    assert e.stats()[2][0] == 1


@pytest.mark.scale
def test_scale_bernoulli_20k_x_60k():
    """n = 20 000 x p = 60 000 dosages on the grid 1/1000 (2.4 GB of codes next to 9.6 GB of FP64), Bernoulli k = 20:
    the FIX16 fit equals the Float64-handle fit."""
    n, p, k, den = 20000, 60000, 20, 1000
    y, z, *_ = synth.simulate_response(2024, n, p, k, "Bernoulli", n_cov=1)
    x = np.empty((n, p), order="F")
    rng = np.random.default_rng(9)
    for j in range(0, p, 5000):
        cols = np.arange(j, min(j + 5000, p))
        g = snp.dosages(synth.packed_columns(2024, n, cols), n) + rng.uniform(-0.05, 0.05, size=(n, cols.size))
        x[:, cols] = np.rint(np.clip(g, 0.0, 2.0) * den) / den
    a = m.fit_iht(y, F16(x, den), z, k=k, d="Bernoulli", l="LogitLink")
    b = m.fit_iht(y, F64(x), z, k=k, d="Bernoulli", l="LogitLink")
    _assert_fits_equal(a, b)
