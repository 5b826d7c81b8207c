"""Dense design matrix without a GPU: the dense oracle against the PLINK oracle, and the host-side argument checks of
B200DenseLinAlg / ihtb_geno_create_dense, which fail before any device is touched."""
import ctypes as C

import numpy as np
import pytest

import mendeliht_jl_b200 as m
from mendeliht_jl_b200 import _lib
from oracle import glm, iht, snp
from oracle.dense import DenseLinAlgOracle


def test_dense_oracle_matches_plink_oracle(normal_data, normal_oracle):
    """A dense matrix holding the standardized genotypes is the PLINK operator (test/wrapper_test.jl:184-206)."""
    d = DenseLinAlgOracle(normal_oracle.dense())
    rng = np.random.default_rng(3)
    v = rng.standard_normal((normal_data["n"], 2)) + 0.5           # not centred
    a, b = d.xt_v(v), normal_oracle.xt_v(v)
    np.testing.assert_allclose(a, b, rtol=1e-12, atol=1e-12 * np.abs(b).max())
    res = iht.fit_iht(normal_data["y"], d, normal_data["z"], k=7, d=glm.NORMAL, l=glm.IDENTITY)
    ref = iht.fit_iht(normal_data["y"], normal_oracle, normal_data["z"], k=7, d=glm.NORMAL, l=glm.IDENTITY)
    assert res.iter == ref.iter
    assert np.array_equal(np.flatnonzero(res.beta), np.flatnonzero(ref.beta))
    assert res.trace.backtracks == ref.trace.backtracks
    np.testing.assert_allclose(res.beta, ref.beta, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(res.c, ref.c, rtol=1e-9, atol=1e-12)
    assert abs(res.logl - ref.logl) <= 1e-9 * abs(ref.logl)


def test_standardize_matches_plink_getindex(normal_data):
    """standardize_genotypes! on integer dosages with missing entries gives SnpLinAlg's getindex bit for bit."""
    n = normal_data["n"]
    codes = snp.unpack_codes(normal_data["bed"][:500], n)
    rng = np.random.default_rng(5)
    codes[rng.random(codes.shape) < 0.02] = 1                       # PLINK code 01 = missing
    bed = snp.pack_codes(codes)
    plink = snp.SnpLinAlgOracle(bed, n)
    dense = DenseLinAlgOracle(snp.dosages(bed, n), standardize=True)
    assert np.array_equal(dense.dense(), plink.dense())
    assert np.array_equal(dense.mu, plink.mu) and np.array_equal(dense.sigma_inv, plink.sigma_inv)
    assert np.array_equal(dense.nmiss, plink.nmiss)


def test_from_array_argument_errors():
    with pytest.raises(m.DimensionMismatch):
        m.B200DenseLinAlg.from_array(np.zeros(10))
    with pytest.raises(m.DimensionMismatch):
        m.B200DenseLinAlg.from_array(np.zeros((2, 3, 4)))
    with pytest.raises(TypeError):
        m.B200DenseLinAlg.from_array(np.zeros((10, 3), dtype=np.int64))
    with pytest.raises(TypeError):
        m.B200DenseLinAlg.from_array(np.zeros((10, 3), dtype=np.float16))
    with pytest.raises(TypeError):
        m.B200DenseLinAlg.from_array([[1.0, 2.0]])
    with pytest.raises(m.DimensionMismatch):
        m.B200DenseLinAlg.from_array(np.zeros((0, 3)))
    with pytest.raises(m.DimensionMismatch):
        m.B200DenseLinAlg.from_array(np.zeros((5, 0), dtype=np.float32))


def test_create_dense_argument_errors():
    """The C entry point validates ld, dtype and standardize before it looks for a device."""
    lib = m.load()
    x = np.zeros((10, 2), order="F")
    h = C.c_void_p()
    xp = C.c_void_p(x.ctypes.data)
    assert lib.ihtb_geno_create_dense(xp, _lib.DENSE_F64, 10, 2, 9, 0, C.byref(h)) == _lib.IHTB_EDIM      # ld < n
    assert lib.ihtb_geno_create_dense(xp, 7, 10, 2, 10, 0, C.byref(h)) == _lib.IHTB_EINVAL               # dtype
    assert lib.ihtb_geno_create_dense(xp, _lib.DENSE_F64, 10, 2, 10, 2, C.byref(h)) == _lib.IHTB_EINVAL  # standardize
    assert lib.ihtb_geno_create_dense(xp, _lib.DENSE_F64, 0, 2, 10, 0, C.byref(h)) == _lib.IHTB_EDIM     # n = 0
    assert lib.ihtb_geno_create_dense(None, _lib.DENSE_F64, 10, 2, 10, 0, C.byref(h)) == _lib.IHTB_EINVAL
    assert lib.ihtb_geno_create_dense_empty(10, 2, 3, 0, C.byref(h)) == _lib.IHTB_EINVAL
    assert not h.value
