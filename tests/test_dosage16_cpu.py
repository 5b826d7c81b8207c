"""16-bit fixed-point dosages without a GPU: the host-side encoding and validation of B200DenseLinAlg.from_dosages,
which fail before any device is touched, and the argument checks of ihtb_geno_create_dosage16."""
import ctypes as C

import numpy as np
import pytest

import mendeliht_jl_b200 as m
from mendeliht_jl_b200 import _lib

DENOMS = [1, 3, 255, 1000, 16384, 32767, 65534]


@pytest.mark.parametrize("den", DENOMS)
def test_round_trip_codes_values_codes(den):
    codes = np.arange(65535, dtype=np.uint16) if den > 2 else np.arange(3, dtype=np.uint16)
    x = (codes.astype(np.float64) / den).reshape(-1, 1)
    assert np.array_equal(m.B200DenseLinAlg.encode_dosages(x, den), codes.reshape(-1, 1))


def test_missing_becomes_the_missing_code_only_when_standardizing():
    x = np.array([[0.0, 1.0], [np.nan, 2.0], [0.5, np.nan]])
    c = m.B200DenseLinAlg.encode_dosages(x, 2, standardize=True)
    assert c.dtype == np.uint16
    assert c.tolist() == [[0, 2], [65535, 4], [1, 65535]]
    with pytest.raises(m.IHTBError) as e:
        m.B200DenseLinAlg.encode_dosages(x, 2)
    assert e.value.code == _lib.IHTB_EDOMAIN and "x[1, 0]" in str(e.value)
    with pytest.raises(m.IHTBError) as e:
        m.B200DenseLinAlg.from_dosages(x, 2)
    assert e.value.code == _lib.IHTB_EDOMAIN


@pytest.mark.parametrize("bad,where", [
    (0.1 + 1e-12, "off the grid"),
    (-0.001, "negative"),
    (65535 / 1000, "above 65534 / D"),
    (np.inf, "infinite"),
    (1.0 / 3.0, "not a multiple of 1/1000"),
])
def test_rejects_entries_that_are_not_codes(bad, where):
    x = np.full((7, 5), 0.25)
    x[4, 2] = bad
    x[6, 3] = bad                                  # later in column-major order: the first one is named
    with pytest.raises(ValueError) as e:
        m.B200DenseLinAlg.from_dosages(x, 1000)
    assert f"x[4, 2] = {bad!r}" in str(e.value), where
    xc = np.ascontiguousarray(x)                   # the layout does not change which entry is named
    with pytest.raises(ValueError) as e:
        m.B200DenseLinAlg.from_dosages(xc, 1000, standardize=True)
    assert "x[4, 2]" in str(e.value)


def test_largest_code_is_accepted_and_the_next_is_not():
    x = np.array([[65534 / 16384]])
    assert m.B200DenseLinAlg.encode_dosages(x, 16384).tolist() == [[65534]]
    with pytest.raises(ValueError):
        m.B200DenseLinAlg.encode_dosages(np.array([[65535 / 16384]]), 16384)


def test_argument_errors():
    x = np.zeros((10, 3))
    for den in (0, -1, 65535, 70000):
        with pytest.raises(ValueError):
            m.B200DenseLinAlg.from_dosages(x, den)
    for den in (2.0, "16384", None, True):
        with pytest.raises(TypeError):
            m.B200DenseLinAlg.from_dosages(x, den)
    for bad in (np.zeros((10, 3), dtype=np.float32), np.zeros((10, 3), dtype=np.int64), np.zeros((10, 3), np.uint16)):
        with pytest.raises(TypeError):
            m.B200DenseLinAlg.from_dosages(bad, 2)
    with pytest.raises(TypeError):
        m.B200DenseLinAlg.from_dosages([[0.5, 1.0]], 2)
    with pytest.raises(m.DimensionMismatch):
        m.B200DenseLinAlg.from_dosages(np.zeros(10), 2)
    with pytest.raises(m.DimensionMismatch):
        m.B200DenseLinAlg.from_dosages(np.zeros((2, 3, 4)), 2)
    with pytest.raises(m.DimensionMismatch):
        m.B200DenseLinAlg.from_dosages(np.zeros((0, 3)), 2)
    with pytest.raises(m.DimensionMismatch):
        m.B200DenseLinAlg.from_dosages(np.zeros((5, 0)), 2)


def test_create_dosage16_argument_errors():
    """The C entry points validate ld, the denominator and standardize before they look for a device, and the float
    constructors keep rejecting the fixed-point storage type, which needs a denominator."""
    lib = m.load()
    codes = np.zeros((10, 2), dtype=np.uint16, order="F")
    cp = codes.ctypes.data_as(C.POINTER(C.c_uint16))
    h = C.c_void_p()
    assert lib.ihtb_geno_create_dosage16(cp, 10, 2, 9, 2, 0, C.byref(h)) == _lib.IHTB_EDIM          # ld < n
    for den in (0, -3, 65535):
        assert lib.ihtb_geno_create_dosage16(cp, 10, 2, 10, den, 0, C.byref(h)) == _lib.IHTB_EINVAL
        assert lib.ihtb_geno_create_dosage16_empty(10, 2, den, 1, C.byref(h)) == _lib.IHTB_EINVAL
    assert lib.ihtb_geno_create_dosage16(cp, 10, 2, 10, 2, 2, C.byref(h)) == _lib.IHTB_EINVAL       # standardize
    assert lib.ihtb_geno_create_dosage16(cp, 0, 2, 10, 2, 0, C.byref(h)) == _lib.IHTB_EDIM          # n = 0
    assert lib.ihtb_geno_create_dosage16(None, 10, 2, 10, 2, 0, C.byref(h)) == _lib.IHTB_EINVAL
    assert lib.ihtb_geno_create_dosage16_empty(10, 0, 2, 0, C.byref(h)) == _lib.IHTB_EDIM
    xp = C.c_void_p(codes.ctypes.data)
    assert lib.ihtb_geno_create_dense(xp, _lib.DENSE_FIX16, 10, 2, 10, 0, C.byref(h)) == _lib.IHTB_EINVAL
    assert lib.ihtb_geno_create_dense_empty(10, 2, _lib.DENSE_FIX16, 0, C.byref(h)) == _lib.IHTB_EINVAL
    assert not h.value
