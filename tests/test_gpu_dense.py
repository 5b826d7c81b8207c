"""Dense design matrices (B200DenseLinAlg, ihtb_geno_create_dense) on the GPU: decode / statistics against the PLINK
handle, X'V and X[:, idx] b against numpy, fits and cross-validation against the dense oracle, PLINK == dense
(test/wrapper_test.jl:184-206), determinism and the rejected cases."""
import ctypes as C

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

DTYPES = [np.float64, np.float32]


def _int_dosages_with_missing(seed, n, p, miss=0.03):
    bed = synth.packed_columns(seed, n, np.arange(p), miss)
    return bed, snp.dosages(bed, n)


def test_decode_and_stats_equal_plink_handle():
    n, p = 1037, 301
    bed, dos = _int_dosages_with_missing(11, n, p)
    g = m.B200SnpLinAlg.from_bed_columns(bed, n)
    d = m.B200DenseLinAlg.from_array(dos, standardize=True)
    a, b = d.decode(), g.decode()
    assert a.view(np.uint64).tolist() == b.view(np.uint64).tolist()          # bit for bit
    for u, v in zip(d.stats(), g.stats()):
        assert np.array_equal(u, v)
    c = m.B200DenseLinAlg.from_array(np.asfortranarray(dos), standardize=True)     # in-place (F order) upload
    assert np.array_equal(c.decode(), b)
    assert np.array_equal(d.decode(100, 200, 7, 50), b[100:200, 7:50])


def test_float32_storage_decodes_exactly():
    rng = np.random.default_rng(2)
    x = rng.standard_normal((77, 45)).astype(np.float32) * 3 + 1
    d = m.B200DenseLinAlg.from_array(x)
    assert np.array_equal(d.decode(), x.astype(np.float64))
    mu, sinv, nm = d.stats()
    assert np.all(mu == 0) and np.all(sinv == 1) and np.all(nm == 0)
    assert d.sweep_stream_bytes() == (77 * 45 * 4, False)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n,p,extra_ld", [(1037, 333, 0), (20, 517, 0), (4099, 130, 13), (2048, 64, 5)])
@pytest.mark.parametrize("mode", [m.SWEEP_FAST, m.SWEEP_EXACT])
def test_xt_v_and_x_support(dtype, n, p, extra_ld, mode):
    rng = np.random.default_rng(n + p)
    big = np.asfortranarray((rng.standard_normal((n + extra_ld, p)) + 3.0).astype(dtype))   # uncentred columns
    x = big[:n]                                                                              # ld = n + extra_ld
    d = m.B200DenseLinAlg.from_array(x)
    xd = x.astype(np.float64)
    for mm in (1, 3, 6):
        V = rng.standard_normal((n, mm)) + 0.7
        out = d.xt_v(V, mode)
        ref = xd.T @ V
        np.testing.assert_allclose(out, ref, rtol=1e-12, atol=1e-12 * np.abs(ref).max())
    v = rng.standard_normal(n) + 2.0
    np.testing.assert_allclose(d.xt_v(v, mode), xd.T @ v, rtol=1e-12, atol=1e-12 * np.abs(xd.T @ v).max())
    o = DenseLinAlgOracle(xd)
    idx = rng.choice(p, size=min(p, 17), replace=False)
    coef = rng.standard_normal(idx.shape[0])
    assert np.array_equal(d.x_support(idx, coef), o.support_xb(idx, coef))       # ascending order, bit for bit
    C2 = rng.standard_normal((idx.shape[0], 2))
    out2 = d.x_support(idx, C2)
    assert np.array_equal(out2[:, 1], o.support_xb(idx, C2[:, 1]))
    c_order = m.B200DenseLinAlg.from_array(np.ascontiguousarray(x))                   # column-block upload
    assert np.array_equal(c_order.decode(), xd)


def _dense_pair(x_raw, dtype):
    x = x_raw.astype(dtype)
    return m.B200DenseLinAlg.from_array(x, standardize=True), DenseLinAlgOracle(x, standardize=True, dtype=dtype)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("cid,d,l,ncov,kw", FIT_CASES, ids=[c[0] for c in FIT_CASES])
def test_fit_matches_dense_oracle(cid, d, l, ncov, kw, dtype):
    seed = 300 + [c[0] for c in FIT_CASES].index(cid)
    y, z, x_raw = case_data(seed, d, ncov)
    g, o = _dense_pair(x_raw, dtype)
    mu, sinv, nm = g.stats()
    np.testing.assert_allclose(mu, o.mu, rtol=1e-14)
    assert np.array_equal(nm, o.nmiss)
    kk = fit_kwargs(kw, P)
    res = m.fit_iht(y, g, z, d=d, l=l, **kk)
    ref = iht.fit_iht(y, o, z, d=d, l=l, **kk)
    assert ref.iter < 200
    compare_fit(res, ref, rtol=1e-5 if kk.get("est_r", "None") != "None" or l not in
                ("IdentityLink", "LogitLink", "LogLink") else 1e-6)
    # both modes run the same FP64 dense sweep: the same model (the IRLS refit of debias may differ in the last bits)
    exact = m.fit_iht(y, g, z, d=d, l=l, sweep_mode=m.SWEEP_EXACT, **kk)
    assert exact.iter == res.iter and [t[1] for t in exact.trace] == [t[1] for t in res.trace]
    assert np.array_equal(np.flatnonzero(exact.beta), np.flatnonzero(res.beta))
    np.testing.assert_allclose(exact.beta, res.beta, rtol=1e-12, atol=0)
    np.testing.assert_allclose(exact.c, res.c, rtol=1e-12, atol=1e-300)


def test_fit_is_deterministic():
    y, z, x_raw = case_data(301, "Bernoulli", 2)
    g, _ = _dense_pair(x_raw, np.float64)
    a = m.fit_iht(y, g, z, k=6, d="Bernoulli", l="LogitLink")
    b = m.fit_iht(y, g, z, k=6, d="Bernoulli", l="LogitLink")
    assert a.beta.tobytes() == b.beta.tobytes() and a.c.tobytes() == b.c.tobytes() and a.trace == b.trace


def _plink_equals_dense(y, z, bed, n, **kw):
    g = m.B200SnpLinAlg.from_bed_columns(bed, n)
    d = m.B200DenseLinAlg.from_array(snp.dosages(bed, n), standardize=True)
    a = m.fit_iht(y, g, z, **kw)
    b = m.fit_iht(y, d, z, **kw)
    assert a.iter == b.iter
    assert np.array_equal(np.flatnonzero(a.beta), np.flatnonzero(b.beta))
    assert [t[1] for t in a.trace] == [t[1] for t in b.trace]
    np.testing.assert_allclose(b.beta, a.beta, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(b.c, a.c, rtol=1e-9, atol=1e-12)
    assert abs(a.logl - b.logl) <= 1e-9 * abs(a.logl)
    assert abs(a.sigma_g - b.sigma_g) <= 1e-9 * abs(a.sigma_g)


def test_plink_equals_dense_normal_bed(normal_data):
    _plink_equals_dense(normal_data["y"], normal_data["z"], normal_data["bed"], normal_data["n"], k=7, d="Normal",
                        l="IdentityLink")


def test_plink_equals_dense_bernoulli_missing():
    n, p = 1500, 3000
    y, z, *_ = synth.simulate_response(77, n, p, 5, "Bernoulli", n_cov=1, missing_rate=0.02)
    bed = synth.packed_columns(77, n, np.arange(p), 0.02)
    _plink_equals_dense(y, z, bed, n, k=5, d="Bernoulli", l="LogitLink")


@pytest.mark.parametrize("dtype", DTYPES)
def test_cv_matches_dense_oracle(dtype):
    y, z, x_raw = case_data(401, "Poisson", 1)
    g, o = _dense_pair(x_raw, dtype)
    folds = synth.folds_for(23, y.shape[0], 3)
    path = [2, 5, 8]
    mses, iters = m.cv_iht(y, g, z, d="Poisson", l="LogLink", path=path, q=3, folds=folds, return_grid=True)
    rm, ri = m.cv_run(y, g, z, folds, 3, path, d="Poisson", l="LogLink")
    _, rgrid, riters = ocv.cv_iht(y, o, z, d="Poisson", l="LogLink", path=path, q=3, folds=folds, return_grid=True)
    assert np.array_equal(iters, riters) and np.array_equal(ri, riters) and riters.max() < 100
    np.testing.assert_allclose(mses, rgrid, rtol=1e-6)
    np.testing.assert_allclose(rm, rgrid, rtol=1e-6)


def test_rejected_cases():
    n, p = 300, 50
    x = continuous_dosages(5, n, p)
    d = m.B200DenseLinAlg.from_array(x, standardize=True)
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
    bad = x.copy()
    bad[3, 4] = np.inf
    with pytest.raises(m.IHTBError) as e:
        m.B200DenseLinAlg.from_array(bad)
    assert e.value.code == _lib.IHTB_EDOMAIN
    bad[3, 4] = np.nan
    with pytest.raises(m.IHTBError) as e:
        m.B200DenseLinAlg.from_array(bad)                      # NaN is only "missing" when standardizing
    assert e.value.code == _lib.IHTB_EDOMAIN
    assert m.B200DenseLinAlg.from_array(bad, standardize=True).stats()[2][4] == np.isnan(x[:, 4]).sum() + 1


@pytest.mark.scale
def test_scale_bernoulli_20k_x_60k():
    """n = 20 000 x p = 60 000 FP64 (9.6 GB on the device), Bernoulli k = 20, against the dense oracle."""
    n, p, k = 20000, 60000, 20
    y, z, *_ = synth.simulate_response(2024, n, p, k, "Bernoulli", n_cov=1)
    x = np.empty((n, p), order="F")
    rng = np.random.default_rng(9)
    for j in range(0, p, 5000):                    # column blocks keep the host copy of the matrix the only big array
        cols = np.arange(j, min(j + 5000, p))
        x[:, cols] = snp.dosages(synth.packed_columns(2024, n, cols), n) + rng.uniform(-0.05, 0.05, size=(n, cols.size))
    g = m.B200DenseLinAlg.from_array(x)
    res = m.fit_iht(y, g, z, k=k, d="Bernoulli", l="LogitLink")
    ref = iht.fit_iht(y, DenseLinAlgOracle(x), z, k=k, d="Bernoulli", l="LogitLink")
    compare_fit(res, ref)
