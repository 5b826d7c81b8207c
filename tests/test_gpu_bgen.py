"""BGEN ingest on the GPU (B200DenseLinAlg.from_bgen, ihtb_geno_load_bgen_columns): bit-for-bit agreement with the
host twin bgen.dosage_codes and with from_dosages / from_array handles of the same codes, the reference's PLINK-vs-BGEN
check on the bundled normal.bed, the iht / cross_validate wrappers, every device-side rejection with the lowest failing
column, determinism, and a 20 000 x 20 000 zlib file."""
import ctypes as C

import numpy as np
import pytest

import mendeliht_jl_b200 as m
from mendeliht_jl_b200 import _lib, bgen, synth
from oracle import snp

import bgen_writer as bw
from dense_cases import continuous_dosages

pytestmark = pytest.mark.gpu

BITS = [1, 3, 8, 12, 15, 16, 23, 32]


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _same_bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape and np.array_equal(_bits(a), _bits(b))


def _write_random(path, n, p, nbits, seed, missing_rate=0.0, compression=1, **kw):
    rng = np.random.default_rng(seed)
    blocks = [bw.random_block(rng, n, nbits, phased=j % 3 == 2, missing_rate=missing_rate) for j in range(p)]
    bw.write(path, blocks, n, compression=compression, **kw)


def _twin_values(path, allele=2):
    codes, miss, bits = bgen.dosage_codes(path, allele)
    x = codes / ((np.int64(1) << bits) - 1).astype(np.float64)
    x[miss] = np.nan
    return codes, miss, bits, x


@pytest.fixture
def small_batches(monkeypatch):
    """More than one inflate batch and more than one device staging batch per load"""
    monkeypatch.setattr(bgen, "INFLATE_BATCH_BYTES", 3000)
    m.load().ihtb_bgen_set_batch_bytes(1000)
    yield
    m.load().ihtb_bgen_set_batch_bytes(0)


# ---- 1. the handle equals the host twin ------------------------------------------------------------------------------------
@pytest.mark.parametrize("nbits", BITS)
@pytest.mark.parametrize("n", [17, 300])
def test_decode_equals_twin(tmp_path, nbits, n, small_batches):
    p = 23
    path = str(tmp_path / "x.bgen")
    _write_random(path, n, p, nbits, seed=nbits * 1000 + n, compression=nbits % 2)
    storages = ["f64"] + (["fix16", "auto"] if nbits <= 15 else ["auto"])
    for allele in (1, 2):
        codes, miss, bits, x = _twin_values(path, allele)
        assert not miss.any()
        for storage in storages:
            h = m.B200DenseLinAlg.from_bgen(path, allele=allele, storage=storage)
            fix = storage == "fix16" or (storage == "auto" and nbits <= 15)
            assert h.dtype == (np.uint16 if fix else np.float64)
            assert h.denominator == ((1 << nbits) - 1 if fix else None)
            _same_bits(h.decode(), x)
            assert len(h.variants) == p and h.samples is None


@pytest.mark.parametrize("nbits", BITS)
def test_missing_standardized_equals_from_array(tmp_path, nbits, small_batches):
    n, p = 531, 19
    path = str(tmp_path / "x.bgen")
    _write_random(path, n, p, nbits, seed=nbits, missing_rate=0.05, sample_ids=[f"id{i}" for i in range(n)])
    codes, miss, bits, x = _twin_values(path)
    assert miss.any()
    ref = m.B200DenseLinAlg.from_array(np.asfortranarray(x), standardize=True)
    for storage in ["f64"] + (["fix16"] if nbits <= 15 else []):
        h = m.B200DenseLinAlg.from_bgen(path, standardize=True, storage=storage)
        assert h.samples == [f"id{i}" for i in range(n)]
        _same_bits(h.decode(), ref.decode())
        for a, b in zip(h.stats(), ref.stats()):
            assert np.array_equal(a, b)


def test_multi_file_concatenation(tmp_path, small_batches):
    n = 70
    paths = [str(tmp_path / f"chr{c}.bgen") for c in range(3)]
    for c, path in enumerate(paths):
        _write_random(path, n, 5 + c, 8, seed=c, sample_ids=[f"s{i}" for i in range(n)] if c != 1 else None)
    h = m.B200DenseLinAlg.from_bgen(paths)
    want = np.hstack([_twin_values(q)[3] for q in paths])
    _same_bits(h.decode(), want)
    assert h.p == 18 and [v.rsid for v in h.variants] == [f"rs{j + 1}" for c in range(3) for j in range(5 + c)]
    assert h.samples == [f"s{i}" for i in range(n)]


# ---- 2. a FIX16 handle from BGEN is the from_dosages handle -------------------------------------------------------------------
@pytest.mark.parametrize("standardize", [False, True])
def test_equals_from_dosages(tmp_path, standardize):
    n, p = 1037, 300
    path = str(tmp_path / "x.bgen")
    _write_random(path, n, p, 8, seed=5, missing_rate=0.02 if standardize else 0.0)
    codes, miss, bits, x = _twin_values(path)
    a = m.B200DenseLinAlg.from_bgen(path, standardize=standardize)
    b = m.B200DenseLinAlg.from_dosages(x, 255, standardize=standardize)
    assert a.denominator == b.denominator == 255
    _same_bits(a.decode(), b.decode())
    for u, v in zip(a.stats(), b.stats()):
        assert np.array_equal(u, v)
    rng = np.random.default_rng(3)
    V = rng.standard_normal((n, 3))
    _same_bits(a.xt_v(V), b.xt_v(V))
    y = x[:, 7].copy()
    y[np.isnan(y)] = 1.0
    cases = [("Normal", "IdentityLink", 0.5 * y + rng.standard_normal(n)),
             ("Bernoulli", "LogitLink", (rng.random(n) < 1 / (1 + np.exp(-(y - 1)))).astype(float)),
             ("Poisson", "LogLink", rng.poisson(np.exp(0.3 * y)).astype(float)),
             ("NegativeBinomial", "LogLink", rng.poisson(np.exp(0.3 * y)).astype(float))]
    for d, l, yy in cases:
        ra = m.fit_iht(yy, a, k=4, d=d, l=l)
        rb = m.fit_iht(yy, b, k=4, d=d, l=l)
        assert ra.iter == rb.iter
        assert np.array_equal(np.flatnonzero(ra.beta), np.flatnonzero(rb.beta))
        _same_bits(ra.beta, rb.beta)
        _same_bits(ra.c, rb.c)
        assert _bits(ra.logl) == _bits(rb.logl)


# ---- 3. the reference's PLINK-vs-BGEN check on normal.bed -----------------------------------------------------------------------
def test_plink_equals_bgen_normal_bed(tmp_path, normal_data):
    y, z, bed, n = normal_data["y"], normal_data["z"], normal_data["bed"], normal_data["n"]
    g = snp.dosages(bed, n)
    path = str(tmp_path / "normal.bgen")
    bw.write(path, [bw.hardcall_block(g[:, j]) for j in range(g.shape[1])], n)
    plink = m.B200SnpLinAlg.from_bed_columns(bed, n)
    d = m.B200DenseLinAlg.from_bgen(path, standardize=True)
    assert d.denominator == 255
    _same_bits(d.decode(), plink.decode())
    a = m.fit_iht(y, plink, z, k=7, d="Normal", l="IdentityLink")
    b = m.fit_iht(y, d, z, k=7, d="Normal", l="IdentityLink")
    assert a.iter == b.iter
    assert np.array_equal(np.flatnonzero(a.beta), np.flatnonzero(b.beta))
    np.testing.assert_allclose(b.beta, a.beta, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(b.c, a.c, rtol=1e-9, atol=1e-12)
    assert abs(a.logl - b.logl) <= 1e-9 * abs(a.logl)


# ---- 4. the file wrappers ---------------------------------------------------------------------------------------------------------
def test_iht_and_cross_validate_on_bgen(tmp_path):
    n, p = 800, 400
    x = np.rint(continuous_dosages(11, n, p, missing_rate=0.0) * 255)
    rng = np.random.default_rng(2)
    blocks = []
    for j in range(p):
        code = x[:, j].astype(np.int64)             # second-allele code: b + 2 c; write a = 0 where possible
        c2 = code // 2
        b = code - 2 * c2
        a = 255 - b - c2
        blocks.append(bw.block(a, b, 8))
    prefix = str(tmp_path / "cohort")
    bw.write(prefix + ".bgen", blocks, n)
    h = m.B200DenseLinAlg.from_bgen(prefix + ".bgen", standardize=True)
    y = 0.8 * h.decode()[:, 5] - 0.6 * h.decode()[:, 40] + rng.standard_normal(n)
    np.savetxt(prefix + "_y.csv", y, delimiter=",")
    ref = m.fit_iht(y, h, np.ones(n), k=3, d="Normal", l="IdentityLink")
    for fn, ph in [(prefix + ".bgen", y), (prefix, prefix + "_y.csv")]:
        r = m.iht(fn, 3, phenotypes=ph)
        assert r.iter == ref.iter and np.array_equal(_bits(r.beta), _bits(ref.beta)) and _bits(r.logl) == _bits(ref.logl)
    folds = synth.folds_for(4, n, 3)
    want = m.cv_iht(y, h, np.ones(n), path=[1, 2, 3], q=3, folds=folds)
    got = m.cross_validate(prefix + ".bgen", path=[1, 2, 3], q=3, phenotypes=y, folds=folds)
    assert np.array_equal(_bits(got), _bits(want))
    Y = np.vstack([y, y])
    with pytest.raises(m.IHTBError, match="multivariate"):
        m.iht(prefix + ".bgen", 3, phenotypes=Y)


# ---- 5. device-side rejections ------------------------------------------------------------------------------------------------------
def _load_raw(blocks, n, den=255, dtype=None, allele=2):
    """(status, message) of one ihtb_geno_load_bgen_columns call on a fresh unfinalized handle"""
    lib = m.load()
    h = C.c_void_p()
    if dtype is None:
        _lib.check(lib.ihtb_geno_create_dosage16_empty(n, len(blocks), den, 1, C.byref(h)))
    else:
        _lib.check(lib.ihtb_geno_create_dense_empty(n, len(blocks), dtype, 1, C.byref(h)))
    try:
        buf = np.frombuffer(b"".join(blocks) + b"\0", dtype=np.uint8)
        offs = np.zeros(len(blocks) + 1, dtype=np.int64)
        np.cumsum([len(b) for b in blocks], out=offs[1:])
        st = lib.ihtb_geno_load_bgen_columns(h, _lib.ptr(buf, C.c_uint8), _lib.ptr(offs, C.c_int64), 0, len(blocks),
                                             allele)
        return st, _lib.last_error()
    finally:
        lib.ihtb_geno_destroy(h)


N = 40
GOOD = bw.block(np.zeros(N, np.int64), np.full(N, 255), 8)
BAD = {
    "n": (bw.block(np.zeros(N + 1, np.int64), np.zeros(N + 1, np.int64), 8), _lib.IHTB_EDIM, "N = 41"),
    "k": (bw.block(np.zeros(N, np.int64), np.zeros(N, np.int64), 8, k=3), _lib.IHTB_EUNSUPPORTED, "3 alleles"),
    "ploidy": (bw.block(np.zeros(N, np.int64), np.zeros(N, np.int64), 8, ploidy=[2] * 9 + [1] + [2] * 30),
               _lib.IHTB_EUNSUPPORTED, "sample 9 is not diploid"),
    "b0": (GOOD[:9 + N] + b"\0" + GOOD[10 + N:], _lib.IHTB_EINVAL, "B = 0"),
    "b33": (GOOD[:9 + N] + b"\x21" + GOOD[10 + N:] + bytes(400), _lib.IHTB_EINVAL, "B = 33"),
    "den": (bw.block(np.zeros(N, np.int64), np.zeros(N, np.int64), 9), _lib.IHTB_EINVAL, "denominator 255"),
    "short": (GOOD[:-1], _lib.IHTB_EINVAL, "shorter than its header \\+ ceil"),
    "header": (GOOD[:20], _lib.IHTB_EINVAL, "shorter than its header"),
    "sum": (bw.block(np.r_[np.zeros(30, np.int64), np.full(10, 200)], np.full(N, 100), 8), _lib.IHTB_EDOMAIN,
            "sample 30: P\\(11\\)"),
}


@pytest.mark.parametrize("case", sorted(BAD))
def test_device_rejections(case):
    blk, code, msg = BAD[case]
    st, err = _load_raw([GOOD, GOOD, blk, GOOD], N)
    assert st == code, err
    assert "block 2 (column 2)" in err
    import re
    assert re.search(msg, err), err


def test_lowest_failing_column_is_reported():
    blocks = [GOOD] * 9
    blocks[7] = BAD["n"][0]
    blocks[3] = BAD["sum"][0]
    blocks[5] = BAD["k"][0]
    for _ in range(3):
        st, err = _load_raw(blocks, N)
        assert st == _lib.IHTB_EDOMAIN and "column 3" in err and "sample 30" in err


def test_rejected_targets():
    st, err = _load_raw([GOOD], N, dtype=_lib.DENSE_F32)
    assert st == _lib.IHTB_EINVAL and "F64" in err
    assert _load_raw([GOOD], N, allele=0)[0] == _lib.IHTB_EINVAL
    st, _ = _load_raw([bw.block(np.zeros(N, np.int64), np.zeros(N, np.int64), 9)], N, dtype=_lib.DENSE_F64)
    assert st == _lib.IHTB_OK                              # Float64 takes any B


def test_mixed_bits(tmp_path):
    path = str(tmp_path / "mixed.bgen")
    rng = np.random.default_rng(0)
    bw.write(path, [bw.random_block(rng, 50, 8), bw.random_block(rng, 50, 8), bw.random_block(rng, 50, 12)], 50)
    with pytest.raises(ValueError, match="rs3.*storage='f64'"):
        m.B200DenseLinAlg.from_bgen(path)
    h = m.B200DenseLinAlg.from_bgen(path, storage="f64")
    _same_bits(h.decode(), _twin_values(path)[3])


def test_missing_without_standardize_fails_at_finalize(tmp_path):
    path = str(tmp_path / "miss.bgen")
    _write_random(path, 64, 4, 8, seed=1, missing_rate=0.2)
    with pytest.raises(m.IHTBError, match="standardize"):
        m.B200DenseLinAlg.from_bgen(path)


# ---- 6. determinism --------------------------------------------------------------------------------------------------------------
def test_deterministic(tmp_path, small_batches):
    path = str(tmp_path / "x.bgen")
    _write_random(path, 999, 61, 8, seed=9, missing_rate=0.03)
    a = m.B200DenseLinAlg.from_bgen(path, standardize=True).decode()
    b = m.B200DenseLinAlg.from_bgen(path, standardize=True).decode()
    _same_bits(a, b)


# ---- 7. scale: 20 000 x 20 000, B = 8, zlib -----------------------------------------------------------------------------------
@pytest.mark.scale
def test_scale_20000(tmp_path):
    n, p, k = 20000, 20000, 10
    rng = np.random.default_rng(20000)
    path = str(tmp_path / "big.bgen")
    blocks = [bw.random_block(rng, n, 8, phased=j % 5 == 4, missing_rate=0.01 if j % 7 == 0 else 0.0)
              for j in range(p)]
    bw.write(path, blocks, n, level=1)
    del blocks
    codes, miss, bits, x = _twin_values(path)
    del codes
    a = m.B200DenseLinAlg.from_bgen(path, standardize=True)
    b = m.B200DenseLinAlg.from_dosages(x, 255, standardize=True)
    causal = rng.choice(p, size=k, replace=False)
    xs = np.where(miss[:, causal], np.nanmean(x[:, causal], axis=0), x[:, causal])
    y = xs @ rng.uniform(0.2, 0.5, size=k) + rng.standard_normal(n)
    del x
    _same_bits(a.decode(0, 200, 0, p), b.decode(0, 200, 0, p))
    ra = m.fit_iht(y, a, k=k, d="Normal", l="IdentityLink")
    rb = m.fit_iht(y, b, k=k, d="Normal", l="IdentityLink")
    assert ra.iter == rb.iter
    assert np.array_equal(np.flatnonzero(ra.beta), np.flatnonzero(rb.beta))
    _same_bits(ra.beta, rb.beta)
    _same_bits(ra.c, rb.c)
    assert _bits(ra.logl) == _bits(rb.logl)
