"""BGEN ingest over a sample and variant selection on the GPU (from_bgen(samples=, sample_file=, variants=),
ihtb_geno_select_bgen_samples): bit-for-bit agreement with the row-mapped host twin over every B, storage and allele,
unsorted rows, phased blocks and several files; identity with the unselected load; equality with from_dosages /
from_array handles of the host subset in decode, stats, fits and CV; missing values and broken variants outside the
selection; the raw C ABI rejections; the file wrappers; determinism; and a 20 000 x 20 000 file."""
import ctypes as C
import re

import numpy as np
import pytest

import mendeliht_jl_b200 as m
from mendeliht_jl_b200 import _lib, bgen, synth

import bgen_writer as bw

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


def _twin_values(path, allele=2, rows=None, cols=None):
    codes, miss, bits = bgen.dosage_codes(path, allele, rows=rows, variants=cols)
    x = codes / ((np.int64(1) << bits) - 1).astype(np.float64)
    x[miss] = np.nan
    return x


def _sample_file(path, ids):
    with open(path, "w") as f:
        f.write("ID_1 ID_2 missing sex\n0 0 0 D\n")
        for s in ids:
            f.write(f"{s} {s} 0 1\n")
    return path


def _same_fit(ra, rb):
    assert ra.iter == rb.iter
    assert np.array_equal(np.flatnonzero(ra.beta), np.flatnonzero(rb.beta))
    _same_bits(ra.beta, rb.beta)
    _same_bits(ra.c, rb.c)
    assert _bits(ra.logl) == _bits(rb.logl)


def _same_stats(a, b):
    for u, v in zip(a.stats(), b.stats()):
        assert np.array_equal(u, v)


@pytest.fixture
def small_batches(monkeypatch):
    """More than one inflate batch and more than one device staging batch per load"""
    monkeypatch.setattr(bgen, "INFLATE_BATCH_BYTES", 3000)
    m.load().ihtb_bgen_set_batch_bytes(1000)
    yield
    m.load().ihtb_bgen_set_batch_bytes(0)


# ---- 1. the selected handle equals the row-mapped twin -----------------------------------------------------------------------
@pytest.mark.parametrize("nbits", BITS)
def test_decode_equals_twin(tmp_path, nbits, small_batches):
    n, p = 300, 23
    path = str(tmp_path / "x.bgen")
    _write_random(path, n, p, nbits, seed=nbits * 7 + 1, compression=nbits % 2)
    rng = np.random.default_rng(nbits)
    rows = rng.permutation(n)[:171]                          # unsorted, 171 of 300
    cols = np.sort(rng.choice(p, size=13, replace=False))    # phased (j % 3 == 2) and unphased blocks
    storages = ["f64"] + (["fix16", "auto"] if nbits <= 15 else ["auto"])
    for allele in (1, 2):
        x = _twin_values(path, allele, rows, cols)
        assert not np.isnan(x).any()
        for storage in storages:
            h = m.B200DenseLinAlg.from_bgen(path, allele=allele, storage=storage, samples=rows.tolist(), variants=cols)
            fix = storage == "fix16" or (storage == "auto" and nbits <= 15)
            assert h.dtype == (np.uint16 if fix else np.float64) and h.shape == (171, 13)
            _same_bits(h.decode(), x)
            assert [v.rsid for v in h.variants] == [f"rs{j + 1}" for j in cols] and h.samples is None


def test_multi_file_ids_and_callable(tmp_path, small_batches):
    n = 70
    ids = [f"s{i}" for i in range(n)]
    paths = [str(tmp_path / f"chr{c}.bgen") for c in range(3)]
    for c, path in enumerate(paths):
        _write_random(path, n, 5 + c, 8, seed=c, sample_ids=ids if c != 1 else None)
    rng = np.random.default_rng(4)
    rows = rng.permutation(n)[:40]
    keep = []
    for q in paths:
        with bgen.BgenFile(q) as f:
            keep += [v.rsid in ("rs1", "rs3", "rs4", "rs7") for v in f.variants]
    cols = np.flatnonzero(keep)
    want = np.hstack([_twin_values(q, rows=rows) for q in paths])[:, cols]
    for variants in (np.array(keep), cols, lambda v: v.rsid in ("rs1", "rs3", "rs4", "rs7")):
        h = m.B200DenseLinAlg.from_bgen(paths, samples=[ids[r] for r in rows], variants=variants)
        _same_bits(h.decode(), want)
        assert h.samples == [ids[r] for r in rows]
        assert [v.rsid for v in h.variants] == ["rs1", "rs3", "rs4"] + ["rs1", "rs3", "rs4"] + ["rs1", "rs3", "rs4", "rs7"]


def test_storage_auto_and_one_b_look_at_kept_variants(tmp_path):
    n = 50
    rng = np.random.default_rng(0)
    path = str(tmp_path / "mixed.bgen")
    bw.write(path, [bw.random_block(rng, n, 16), bw.random_block(rng, n, 8), bw.random_block(rng, n, 12),
                    bw.random_block(rng, n, 8)], n)
    h = m.B200DenseLinAlg.from_bgen(path, variants=[1, 3])
    assert h.denominator == 255
    _same_bits(h.decode(), _twin_values(path, cols=[1, 3]))
    with pytest.raises(ValueError, match="storage='f64'"):
        m.B200DenseLinAlg.from_bgen(path, variants=[1, 2])


# ---- 2. identity: selecting every sample in order is the unselected load -------------------------------------------------------
def test_identity_selection(tmp_path, small_batches):
    n, p = 517, 40
    path = str(tmp_path / "x.bgen")
    _write_random(path, n, p, 8, seed=3, missing_rate=0.03)
    for storage in ("fix16", "f64"):
        a = m.B200DenseLinAlg.from_bgen(path, standardize=True, storage=storage)
        b = m.B200DenseLinAlg.from_bgen(path, standardize=True, storage=storage, samples=range(n))
        _same_bits(a.decode(), b.decode())
        _same_stats(a, b)
        y = a.decode()[:, 4] - 0.5 * a.decode()[:, 11] + np.random.default_rng(1).standard_normal(n)
        _same_fit(m.fit_iht(y, a, k=3, d="Normal", l="IdentityLink"), m.fit_iht(y, b, k=3, d="Normal", l="IdentityLink"))


# ---- 3. a selected, standardized handle equals the handle of the host subset ----------------------------------------------------
@pytest.mark.parametrize("storage", ["fix16", "f64"])
def test_equals_host_subset(tmp_path, storage, small_batches):
    n, p = 1037, 120
    path = str(tmp_path / "x.bgen")
    _write_random(path, n, p, 8, seed=5, missing_rate=0.02)
    rng = np.random.default_rng(6)
    rows = rng.permutation(n)[:700]
    cols = np.flatnonzero(rng.random(p) < 0.6)
    x = _twin_values(path, rows=rows, cols=cols)
    a = m.B200DenseLinAlg.from_bgen(path, standardize=True, storage=storage, samples=rows, variants=cols)
    b = m.B200DenseLinAlg.from_dosages(x, 255, standardize=True) if storage == "fix16" else \
        m.B200DenseLinAlg.from_array(np.asfortranarray(x), standardize=True)
    _same_bits(a.decode(), b.decode())
    _same_stats(a, b)
    xs = b.decode()
    nn = rows.shape[0]
    y = 0.7 * xs[:, 3] - 0.5 * xs[:, 30] + 0.4 * xs[:, 50] + rng.standard_normal(nn)
    _same_fit(m.fit_iht(y, a, k=4, d="Normal", l="IdentityLink"), m.fit_iht(y, b, k=4, d="Normal", l="IdentityLink"))
    folds = synth.folds_for(8, nn, 3)
    ga = m.cv_iht(y, a, np.ones(nn), path=[1, 2, 3, 4], q=3, folds=folds)
    gb = m.cv_iht(y, b, np.ones(nn), path=[1, 2, 3, 4], q=3, folds=folds)
    _same_bits(ga, gb)


# ---- 4. missing values and broken variants outside the selection ---------------------------------------------------------------
def test_missing_only_in_dropped_rows(tmp_path):
    n, p = 64, 6
    rng = np.random.default_rng(2)
    miss = np.zeros(n, dtype=bool)
    miss[[3, 10, 40]] = True
    blocks = [bw.block(np.zeros(n, np.int64), rng.integers(0, 256, n), 8, missing=miss) for _ in range(p)]
    path = str(tmp_path / "miss.bgen")
    bw.write(path, blocks, n)
    kept = [i for i in range(n) if not miss[i]][::-1]
    for storage in ("fix16", "f64"):
        h = m.B200DenseLinAlg.from_bgen(path, storage=storage, samples=kept)
        _same_bits(h.decode(), _twin_values(path, rows=kept))
        with pytest.raises(m.IHTBError, match="standardize"):
            m.B200DenseLinAlg.from_bgen(path, storage=storage, samples=kept + [10])


def test_dropped_broken_variants_are_never_read(tmp_path):
    n = 30
    rng = np.random.default_rng(1)
    good = [bw.random_block(rng, n, 8) for _ in range(4)]
    path = str(tmp_path / "broken.bgen")
    bw.write(path, [good[0], good[1], bw.block(np.zeros(n, np.int64), np.zeros(n, np.int64), 8, k=3), good[2],
                    good[3]], n)
    data = bytearray(open(path, "rb").read())
    with bgen.BgenFile(path) as f:
        pos = int(f._data_pos[1])
    data[pos + 2] ^= 0xFF                                      # variant 1: corrupt zlib data
    open(path, "wb").write(bytes(data))
    with pytest.raises(ValueError, match="corrupt zlib"):
        m.B200DenseLinAlg.from_bgen(path)
    with pytest.raises(ValueError, match="corrupt zlib"):
        m.B200DenseLinAlg.from_bgen(path, variants=[0, 1])
    h = m.B200DenseLinAlg.from_bgen(path, variants=[0, 3, 4])
    _same_bits(h.decode(), _twin_values(path, cols=[0, 3, 4]))


# ---- 5. the raw C ABI --------------------------------------------------------------------------------------------------------------
N = 40
GOOD = bw.block(np.zeros(N, np.int64), np.full(N, 255), 8)


def _handle(n, p, den=255, dtype=None, standardize=1):
    lib = m.load()
    h = C.c_void_p()
    if dtype is None:
        _lib.check(lib.ihtb_geno_create_dosage16_empty(n, p, den, standardize, C.byref(h)))
    else:
        _lib.check(lib.ihtb_geno_create_dense_empty(n, p, dtype, standardize, C.byref(h)))
    return h


def _select(h, rows, n_file):
    r = np.ascontiguousarray(rows, dtype=np.int64)
    st = m.load().ihtb_geno_select_bgen_samples(h, _lib.ptr(r, C.c_int64), n_file)
    return st, _lib.last_error()


def _load(h, blocks, j_first=0):
    buf = np.frombuffer(b"".join(blocks) + b"\0", dtype=np.uint8)
    offs = np.zeros(len(blocks) + 1, dtype=np.int64)
    np.cumsum([len(b) for b in blocks], out=offs[1:])
    st = m.load().ihtb_geno_load_bgen_columns(h, _lib.ptr(buf, C.c_uint8), _lib.ptr(offs, C.c_int64), j_first,
                                              len(blocks), 2)
    return st, _lib.last_error()


def _selected_load(blocks, rows, n_file=N, dtype=None):
    h = _handle(len(rows), len(blocks), dtype=dtype)
    try:
        st, err = _select(h, rows, n_file)
        assert st == _lib.IHTB_OK, err
        return _load(h, blocks)
    finally:
        m.load().ihtb_geno_destroy(h)


def test_select_where_allowed():
    lib = m.load()
    h = _handle(10, 2)
    try:                                                       # after a load
        assert _load(h, [bw.block(np.zeros(10, np.int64), np.zeros(10, np.int64), 8)])[0] == _lib.IHTB_OK
        st, err = _select(h, range(10), 20)
        assert st == _lib.IHTB_EINVAL and "already loaded" in err
    finally:
        lib.ihtb_geno_destroy(h)
    h = _handle(10, 2, dtype=_lib.DENSE_F32)
    try:
        st, err = _select(h, range(10), 20)
        assert st == _lib.IHTB_EINVAL and "F64" in err
    finally:
        lib.ihtb_geno_destroy(h)
    h = C.c_void_p()
    _lib.check(lib.ihtb_geno_create_empty(10, 2, 1, 1, 1, C.byref(h)))
    try:
        st, err = _select(h, range(10), 20)
        assert st == _lib.IHTB_EINVAL and "not a dense handle" in err
    finally:
        lib.ihtb_geno_destroy(h)
    fin = m.B200DenseLinAlg.from_array(np.ones((10, 2)))
    st, err = _select(fin._h, range(10), 20)
    assert st == _lib.IHTB_EINVAL and "finalized" in err
    for dtype in (None, _lib.DENSE_F64):                       # a second selection before any load replaces the first
        h = _handle(3, 1, dtype=dtype, standardize=0)
        try:
            assert _select(h, [0, 1, 2], N)[0] == _lib.IHTB_OK
            assert _select(h, [39, 0, 7], N)[0] == _lib.IHTB_OK
            # file sample i: (a, b) = (0, i), second-allele code 510 - i
            assert _load(h, [bw.block(np.zeros(N, np.int64), np.arange(N), 8)])[0] == _lib.IHTB_OK
            _lib.check(lib.ihtb_geno_finalize(h))
            out = np.zeros(3)
            _lib.check(lib.ihtb_geno_decode(h, 0, 3, 0, 1, _lib.ptr(out, C.c_double)))
            assert out.tolist() == [471 / 255, 510 / 255, 503 / 255]
        finally:
            lib.ihtb_geno_destroy(h)


@pytest.mark.parametrize("rows,n_file,msg", [
    ([0, 5, 3, 5, 1], N, r"rows\[1\] and rows\[3\] are both file sample 5"),
    ([2, 9, 9, 2, 4], N, r"rows\[1\] and rows\[2\] are both file sample 9"),
    ([0, 1, 40, 2, 3], N, r"rows\[2\] = 40 is outside \[0, n_file = 40\)"),
    ([0, 1, 2, -1, 3], N, r"rows\[3\] = -1"),
    ([0, 1, 2, 3, 4], 4, "n_file = 4"),
    ([0, 1, 2, 3, 4], 1 << 32, "n_file = 4294967296"),
])
def test_select_rejects_rows(rows, n_file, msg):
    h = _handle(len(rows), 1)
    try:
        st, err = _select(h, rows, n_file)
        assert st == _lib.IHTB_EINVAL and re.search(msg, err), err
    finally:
        m.load().ihtb_geno_destroy(h)


def test_block_n_must_be_n_file():
    st, err = _selected_load([GOOD, bw.block(np.zeros(N - 1, np.int64), np.zeros(N - 1, np.int64), 8)], [3, 1, 2],
                             n_file=N)
    assert st == _lib.IHTB_EDIM and "column 1" in err and "N = 39" in err and "n_file = 40" in err, err
    st, err = _selected_load([GOOD], [3, 1, 2], n_file=N + 1)
    assert st == _lib.IHTB_EDIM and "n_file = 41" in err, err


@pytest.mark.parametrize("dtype", [None, _lib.DENSE_F64])
def test_kept_samples_only_are_checked(dtype):
    ploidy = bw.block(np.zeros(N, np.int64), np.zeros(N, np.int64), 8, ploidy=[2] * 9 + [1] + [2] * 30)
    total = bw.block(np.r_[np.zeros(30, np.int64), np.full(10, 200)], np.full(N, 100), 8)
    st, err = _selected_load([GOOD, ploidy], [12, 9, 0], dtype=dtype)
    assert st == _lib.IHTB_EUNSUPPORTED and "column 1" in err and "file sample 9 is not diploid" in err, err
    st, err = _selected_load([GOOD, total], [1, 35, 33, 2], dtype=dtype)
    assert st == _lib.IHTB_EDOMAIN and "file sample 33" in err, err
    rows = [12, 0, 29, 8, 10]                                  # neither file sample 9 nor 30..39
    assert _selected_load([GOOD, ploidy, total], rows, dtype=dtype)[0] == _lib.IHTB_OK


def test_lowest_failing_column_is_reported():
    k3 = bw.block(np.zeros(N, np.int64), np.zeros(N, np.int64), 8, k=3)
    total = bw.block(np.r_[np.zeros(30, np.int64), np.full(10, 200)], np.full(N, 100), 8)
    blocks = [GOOD] * 9
    blocks[7] = bw.block(np.zeros(N + 1, np.int64), np.zeros(N + 1, np.int64), 8)
    blocks[3] = total
    blocks[5] = k3
    for _ in range(2):
        st, err = _selected_load(blocks, list(range(39, 14, -1)))
        assert st == _lib.IHTB_EDOMAIN and "column 3" in err and "file sample 30" in err, err
    st, err = _selected_load(blocks, list(range(20)))          # block 3 is fine on these rows
    assert st == _lib.IHTB_EUNSUPPORTED and "column 5" in err and "3 alleles" in err, err


# ---- 6. the file wrappers ----------------------------------------------------------------------------------------------------------
def test_iht_and_cross_validate_with_selection(tmp_path):
    n, p = 800, 300
    ids = [f"{1000000 + 7 * i}" for i in range(n)]
    prefix = str(tmp_path / "cohort")
    _write_random(prefix + ".bgen", n, p, 8, seed=12, missing_rate=0.01)
    sf = _sample_file(prefix + ".sample", ids)
    rng = np.random.default_rng(3)
    keep = [ids[i] for i in rng.permutation(n)[:550]]
    cols = np.flatnonzero(rng.random(p) < 0.7)
    h = m.B200DenseLinAlg.from_bgen(prefix + ".bgen", standardize=True, samples=keep, sample_file=sf, variants=cols)
    assert h.samples == keep
    xs = h.decode()
    y = 0.8 * xs[:, 5] - 0.6 * xs[:, 40] + rng.standard_normal(len(keep))
    ref = m.fit_iht(y, h, np.ones(len(keep)), k=3, d="Normal", l="IdentityLink")
    r = m.iht(prefix + ".bgen", 3, phenotypes=y, samples=keep, sample_file=sf, variants=cols)
    _same_fit(r, ref)
    folds = synth.folds_for(4, len(keep), 3)
    want = m.cv_iht(y, h, np.ones(len(keep)), path=[1, 2, 3], q=3, folds=folds)
    got = m.cross_validate(prefix, path=[1, 2, 3], q=3, phenotypes=y, folds=folds, samples=keep, sample_file=sf,
                           variants=cols)
    _same_bits(got, want)


# ---- 7. determinism ----------------------------------------------------------------------------------------------------------------
def test_deterministic(tmp_path, small_batches):
    n = 999
    path = str(tmp_path / "x.bgen")
    _write_random(path, n, 61, 8, seed=9, missing_rate=0.03)
    rows = np.random.default_rng(0).permutation(n)[:600]
    a = m.B200DenseLinAlg.from_bgen(path, standardize=True, samples=rows, variants=lambda v: v.pos % 2 == 0)
    b = m.B200DenseLinAlg.from_bgen(path, standardize=True, samples=rows, variants=lambda v: v.pos % 2 == 0)
    _same_bits(a.decode(), b.decode())
    _same_stats(a, b)


# ---- 8. scale: 20 000 x 20 000, B = 8, zlib; 12 000 shuffled samples and half of the variants -------------------------------
@pytest.mark.scale
def test_scale_20000(tmp_path):
    n, p, k = 20000, 20000, 10
    rng = np.random.default_rng(20001)
    path = str(tmp_path / "big.bgen")
    blocks = [bw.random_block(rng, n, 8, phased=j % 5 == 4, missing_rate=0.01 if j % 7 == 0 else 0.0)
              for j in range(p)]
    bw.write(path, blocks, n, level=1)
    del blocks
    rows = rng.permutation(n)[:12000]
    cols = np.sort(rng.choice(p, size=p // 2, replace=False))
    x = _twin_values(path, rows=rows, cols=cols)
    a = m.B200DenseLinAlg.from_bgen(path, standardize=True, samples=rows, variants=cols)
    b = m.B200DenseLinAlg.from_dosages(x, 255, standardize=True)
    causal = rng.choice(cols.shape[0], size=k, replace=False)
    xc = x[:, causal]
    xs = np.where(np.isnan(xc), np.nanmean(xc, axis=0), xc)
    y = xs @ rng.uniform(0.2, 0.5, size=k) + rng.standard_normal(rows.shape[0])
    del x
    _same_bits(a.decode(0, 200, 0, a.p), b.decode(0, 200, 0, b.p))
    _same_stats(a, b)
    _same_fit(m.fit_iht(y, a, k=k, d="Normal", l="IdentityLink"), m.fit_iht(y, b, k=k, d="Normal", l="IdentityLink"))
