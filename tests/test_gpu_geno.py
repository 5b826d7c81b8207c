"""GPU parity of the genotype operator (SnpLinAlg replacement) against the CPU oracle, through the C ABI."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import mendeliht_jl_b200 as m
from mendeliht_jl_b200 import synth
from oracle import snp


@pytest.mark.parametrize("n,p,miss", [(1000, 257, 0.0), (1003, 300, 0.02), (515, 64, 0.3), (7, 5, 0.0), (2049, 130, 0.001)])
def test_stats_decode_packed_bit_exact(n, p, miss):
    bed = synth.packed_columns(11, n, np.arange(p), miss)
    g = m.B200SnpLinAlg.from_bed_columns(bed, n)
    o = snp.SnpLinAlgOracle(bed, n)
    mu, sinv, nm = g.stats()
    assert np.array_equal(nm, o.nmiss)
    assert np.array_equal(mu, o.mu)                 # integer counts, one IEEE division: bit-exact
    assert np.array_equal(sinv, o.sigma_inv)
    assert np.array_equal(g.decode(), o.dense())    # decoded genotypes bit-exact
    assert np.array_equal(g.decode(3, min(n, 40), 1, min(p, 9)), o.dense()[3:min(n, 40), 1:min(p, 9)])
    assert np.array_equal(g.packed(), bed)


def test_device_generator_matches_numpy_twin():
    for n, p, miss, j0 in [(1003, 200, 0.0, 0), (2500, 150, 0.01, 1000)]:
        g = m.B200SnpLinAlg.synthetic(n, p, 2024, miss, j0)
        assert np.array_equal(g.packed(), synth.packed_columns(2024, n, np.arange(j0, j0 + p), miss))


@pytest.mark.parametrize("n,p,miss", [(1000, 300, 0.0), (1003, 513, 0.01), (4099, 260, 0.0), (600, 129, 0.2)])
def test_xt_v_exact_and_fast(n, p, miss):
    bed = synth.packed_columns(5, n, np.arange(p), miss)
    g = m.B200SnpLinAlg.from_bed_columns(bed, n)
    o = snp.SnpLinAlgOracle(bed, n)
    rng = np.random.default_rng(0)
    v = rng.normal(size=n) + 0.3
    ref = o.xt_v(v)
    scale = np.abs(ref).max()
    ex = g.xt_v(v, m.SWEEP_EXACT)
    np.testing.assert_allclose(ex, ref, rtol=0, atol=1e-11 * scale)      # FP64: stated tolerance 1e-6 rel, we see ~1e-14
    fa = g.xt_v(v, m.SWEEP_FAST)
    # FP32-accumulate class (north_star tolerance 1e-4 relative); the proven bound is 2^-18 * ||v - mean||_1 * sinv
    bound = (2.0 ** -18) * np.abs(v - v.mean()).sum() * o.sigma_inv
    assert np.all(np.abs(fa - ref) <= bound + 1e-12 * scale)
    assert np.max(np.abs(fa - ref)) < 1e-4 * scale
    # multi right-hand sides (MvNormal skinny X'R)
    V = rng.normal(size=(n, 3))
    np.testing.assert_allclose(g.xt_v(V, m.SWEEP_EXACT), o.xt_v(V), rtol=0, atol=1e-11 * np.abs(o.xt_v(V)).max())
    # linearity (size-independent property)
    a = g.xt_v(v, m.SWEEP_EXACT); b = g.xt_v(2 * v + 1.0, m.SWEEP_EXACT)
    np.testing.assert_allclose(b, 2 * a, rtol=0, atol=1e-10 * scale)    # centring kills the constant
    # pair sweep (two right-hand sides per pass, half2 tables): proven bound 2^-8 * ||v - mean||_1 * sinv per entry;
    # right-hand sides of very different magnitude exercise the per-vector power-of-two scaling
    V5 = rng.normal(size=(n, 5)) * np.array([1.0, 1e-6, 3e4, 0.02, 7.0]) + np.array([0.0, 1.0, -5.0, 0.0, 2.0])
    got, want = g.xt_v(V5, m.SWEEP_PAIR), o.xt_v(V5)
    # the bound the fits use: 3.1 * 2^-11 * ||u||_2 * sinv_j * max(sqrt(sum_i g_ij^2), 1)  (Cauchy-Schwarz on the
    # absolute dot product every FP16 rounding is relative to); the last, odd vector takes the FP32 tables
    gn = np.maximum(np.sqrt((np.where(np.isnan(snp.dosages(bed, n)), 0.0, snp.dosages(bed, n)) ** 2).sum(axis=0)), 1.0)
    for t in range(5):
        u = V5[:, t] - V5[:, t].mean()
        bnd = (3.1 * 2.0 ** -11 if t < 4 else 2.0 ** -20) * np.sqrt((u ** 2).sum()) * o.sigma_inv * gn
        assert np.all(np.abs(got[:, t] - want[:, t]) <= bnd + 1e-12 * np.abs(want[:, t]).max()), t
        assert np.all(np.abs(got[:, t] - want[:, t]) <= (2.0 ** -8) * np.abs(u).sum() * o.sigma_inv + 1e-12 * np.abs(want[:, t]).max())
    assert np.array_equal(g.xt_v(V5[:, :1], m.SWEEP_PAIR), g.xt_v(V5[:, :1], m.SWEEP_FAST))   # odd one out: FAST
    zero = np.zeros((n, 2)); zero[:, 1] = 3.0                      # constant vectors: u = 0, scale falls back to 1
    assert np.all(g.xt_v(zero, m.SWEEP_PAIR) == 0.0)


@pytest.mark.parametrize("n,p,miss", [(1003, 513, 0.01), (640, 9, 0.0), (641, 130, 0.3), (3200, 257, 0.0), (50, 4, 0.0),
                                      (12801, 1030, 0.002)])
def test_ternary_copy_sweeps(n, p, miss):
    """The FAST / PAIR sweeps stream a ternary copy of the tiles (five dosages per byte, 640 samples per 128-byte chunk,
    common.cuh): same error bounds against the oracle as the 2-bit stream, everything else reads the PLINK codes."""
    bed = synth.packed_columns(6, n, np.arange(p), miss)
    o = snp.SnpLinAlgOracle(bed, n)
    hs = {}
    for flag in ("1", "0"):
        os.environ["IHTB_TERN"] = flag
        try:
            hs[flag] = m.B200SnpLinAlg.from_bed_columns(bed, n)
        finally:
            os.environ.pop("IHTB_TERN", None)
    p4 = (p + 3) // 4 * 4
    assert hs["1"].sweep_stream_bytes() == (-(-n // 640) * 128 * p4, True)
    assert hs["0"].sweep_stream_bytes() == (-(-n // 512) * 128 * p4, False)
    rng = np.random.default_rng(1)
    V = rng.normal(size=(n, 3)) * np.array([1.0, 40.0, 1e-3]) + np.array([0.3, -2.0, 0.0])
    want = o.xt_v(V)
    dos = snp.dosages(bed, n)
    gn = np.maximum(np.sqrt((np.where(np.isnan(dos), 0.0, dos) ** 2).sum(axis=0)), 1.0)
    for flag, g in hs.items():
        assert np.array_equal(g.packed(), bed) and np.array_equal(g.decode(), o.dense())
        for t in range(3):
            u = V[:, t] - V[:, t].mean()
            tiny = 1e-12 * np.abs(want[:, t]).max()
            fa = g.xt_v(V[:, t], m.SWEEP_FAST)
            assert np.all(np.abs(fa - want[:, t]) <= (2.0 ** -18) * np.abs(u).sum() * o.sigma_inv + tiny), (flag, t)
            assert np.all(np.abs(fa - want[:, t]) <= (2.0 ** -20) * np.sqrt((u ** 2).sum()) * o.sigma_inv * gn + tiny), (flag, t)
        got = g.xt_v(V, m.SWEEP_PAIR)
        for t in range(3):
            u = V[:, t] - V[:, t].mean()
            bnd = (3.1 * 2.0 ** -11 if t < 2 else 2.0 ** -20) * np.sqrt((u ** 2).sum()) * o.sigma_inv * gn
            assert np.all(np.abs(got[:, t] - want[:, t]) <= bnd + 1e-12 * np.abs(want[:, t]).max()), (flag, t)
    assert np.array_equal(hs["1"].xt_v(V, m.SWEEP_EXACT), hs["0"].xt_v(V, m.SWEEP_EXACT))     # FP64 path: the PLINK tiles
    for g in hs.values():
        g.close()


def test_x_support_bit_exact():
    n, p = 1003, 400
    bed = synth.packed_columns(9, n, np.arange(p), 0.01)
    g = m.B200SnpLinAlg.from_bed_columns(bed, n)
    o = snp.SnpLinAlgOracle(bed, n)
    rng = np.random.default_rng(1)
    idx = np.sort(rng.permutation(p)[:37])
    coef = rng.normal(size=37)
    # same formula, same order of additions as the reference's getindex loop: bit-exact
    assert np.array_equal(g.x_support(idx, coef), o.support_xb(idx, coef))
    C = rng.normal(size=(37, 5))
    got = g.x_support(idx, C)
    for t in range(5):
        assert np.array_equal(got[:, t], o.support_xb(idx, C[:, t]))
    assert np.array_equal(g.x_support(np.zeros(0, np.int64), np.zeros(0)), np.zeros(n))


def test_bundled_fixture_sweep(normal_data, normal_oracle):
    g = m.B200SnpLinAlg.from_bed_columns(normal_data["bed"], normal_data["n"])
    r = normal_data["y"] - normal_data["y"].mean()
    ref = normal_oracle.xt_v(r)
    np.testing.assert_allclose(g.xt_v(r, m.SWEEP_EXACT), ref, rtol=0, atol=1e-10)
    np.testing.assert_allclose(g.xt_v(r, m.SWEEP_FAST), ref, rtol=0, atol=1e-4 * np.abs(ref).max())


def test_fast_sweep_matches_exact_at_scale():
    """BASELINE-size property check (the oracle cannot hold this matrix): the FAST sweep stays inside its proven
    error bound of the EXACT sweep for every column, repeatedly (catches pipeline races that small cases miss)."""
    n, p = 50000, 200000
    g = m.B200SnpLinAlg.synthetic(n, p, 2024)
    _, sinv, _ = g.stats()
    rng = np.random.default_rng(3)
    for rep in range(4):
        v = rng.normal(size=n) * (1 + rep) + 0.1 * rep
        ex = g.xt_v(v, m.SWEEP_EXACT)
        fa = g.xt_v(v, m.SWEEP_FAST)
        bound = (2.0 ** -18) * np.abs(v - v.mean()).sum() * sinv
        assert np.all(np.abs(fa - ex) <= bound + 1e-9 * np.abs(ex).max())
        v2 = rng.normal(size=n) * 0.01
        pr = g.xt_v(np.stack([v, v2], axis=1), m.SWEEP_PAIR)
        cnt = g.counts()
        sgn = sinv * np.maximum(np.sqrt(cnt[2] + 4.0 * cnt[3]), 1.0)
        assert np.all(np.abs(pr[:, 0] - ex) <= 3.1 * 2.0 ** -11 * np.linalg.norm(v - v.mean()) * sgn)
        assert np.all(np.abs(pr[:, 1] - g.xt_v(v2, m.SWEEP_EXACT)) <= 3.1 * 2.0 ** -11 * np.linalg.norm(v2 - v2.mean()) * sgn)
    # checksum of checksums against a column subsample computed by the numpy twin of the generator
    cols = np.sort(rng.permutation(p)[:64])
    xs = synth.standardized_columns(2024, n, cols)
    np.testing.assert_allclose(ex[cols], xs.T @ v, rtol=0, atol=1e-8 * np.abs(ex).max())


def test_errors():
    with pytest.raises(m.DimensionMismatch):
        m.B200SnpLinAlg.from_bed_columns(np.zeros((4, 2), dtype=np.uint8), 100)   # stride < ceil(n/4)
    g = m.B200SnpLinAlg.synthetic(100, 10, 1)
    with pytest.raises(m.DimensionMismatch):
        g.decode(0, 101, 0, 1)
    with pytest.raises(m.DimensionMismatch):
        g.x_support(np.array([10]), np.array([1.0]))


def test_counts_maf_and_piecewise_ingest(tmp_path):
    """SnpArrays counts/maf (SURVEY.md 8f2) and ingest from several .bed files == ingest of the concatenation."""
    n, p, miss = 1003, 777, 0.02
    bed = synth.packed_columns(5, n, np.arange(p), miss)
    g = m.B200SnpLinAlg.from_bed_columns(bed, n)
    codes = np.stack([(bed >> (2 * s)) & 3 for s in range(4)], axis=2).reshape(p, -1)[:, :n]
    cnt = np.stack([(codes == c).sum(axis=1) for c in range(4)])
    np.testing.assert_array_equal(g.counts(), cnt)
    nobs = n - cnt[1]
    f = (cnt[2] + 2 * cnt[3]) / (2 * nobs)
    np.testing.assert_array_equal(g.maf(), np.where(f > 0.5, 1 - f, f))
    # three "chromosomes" of unequal size, written as real .bed files
    cuts = [0, 300, 301, p]
    paths = []
    for a, b in zip(cuts[:-1], cuts[1:]):
        path = tmp_path / f"chr{a}.bed"
        with open(path, "wb") as fh:
            fh.write(bytes([0x6C, 0x1B, 0x01])); fh.write(bed[a:b].tobytes())
        paths.append(str(path))
    g2 = m.B200SnpLinAlg.from_bed_files(paths, n)
    assert g2.shape == (n, p)
    np.testing.assert_array_equal(g2.packed(), g.packed())
    for a, b in zip(g2.stats(), g.stats()):
        np.testing.assert_array_equal(a, b)
    v = np.random.default_rng(0).normal(size=n)
    np.testing.assert_array_equal(g2.xt_v(v, m.SWEEP_EXACT), g.xt_v(v, m.SWEEP_EXACT))
    # a handle that is not finalized refuses to compute
    lib = m.load()
    import ctypes as C
    h = C.c_void_p()
    m._lib.check(lib.ihtb_geno_create_empty(n, p, 1, 1, 1, C.byref(h)))
    mu = np.empty(p)
    assert lib.ihtb_geno_stats(h, mu.ctypes.data_as(C.POINTER(C.c_double)), None, None) == m._lib.IHTB_EINVAL
    bedc = np.ascontiguousarray(bed)
    m._lib.check(lib.ihtb_geno_load_columns(h, bedc.ctypes.data_as(C.POINTER(C.c_uint8)), bedc.shape[1], 0, p))
    m._lib.check(lib.ihtb_geno_finalize(h))
    assert lib.ihtb_geno_finalize(h) == m._lib.IHTB_EINVAL
    m._lib.check(lib.ihtb_geno_stats(h, mu.ctypes.data_as(C.POINTER(C.c_double)), None, None))
    np.testing.assert_array_equal(mu, g.stats()[0])
    lib.ihtb_geno_destroy(h)
    with pytest.raises(ValueError):
        bad = tmp_path / "bad.bed"
        bad.write_bytes(b"\x00\x00\x00" + bed[:2].tobytes())
        m.B200SnpLinAlg.from_bed_files([str(bad)], n)


@pytest.mark.parametrize("n,p,miss,ncols", [(1003, 300, 0.05, 257), (5000, 64, 0.0, 64), (513, 40, 0.3, 9), (40000, 128, 0.001, 500)])
def test_nibble_gather_matches_decode_kernel(n, p, miss, ncols):
    """Exact re-scoring of candidate columns: the nibble-table kernel (one right-hand side, every univariate fit) against the
    per-column decode kernel, with missing data (CSR imputation term) and ragged n."""
    g = m.B200SnpLinAlg.synthetic(n, p, 77, miss)
    ms, err = g.gather_bench(ncols, 1)
    assert err <= 1e-13, err
    g.close()


@pytest.mark.parametrize("n,p,miss", [(640, 8, 0.0), (1003, 13, 0.05), (2500, 130, 0.2)])
def test_ternary_tiles_match_host_twin(n, p, miss):
    """The ternary copy as it lies in HBM equals the numpy restatement of its format byte for byte."""
    bed = synth.packed_columns(9, n, np.arange(p), miss)
    os.environ["IHTB_TERN"] = "1"
    try:
        g = m.B200SnpLinAlg.from_bed_columns(bed, n)
    finally:
        os.environ.pop("IHTB_TERN", None)
    assert np.array_equal(g.ternary_tiles(), synth.ternary_tiles(bed, n))
    g.close()
