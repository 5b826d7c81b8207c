"""Sample and variant selection of BGEN input on the host (no GPU): Oxford .sample files, the row-mapped host twin,
batching over kept variants only, every argument error of from_bgen's samples / sample_file / variants (raised before
the library is touched), and how iht / cross_validate forward the selection keywords."""
import numpy as np
import pytest

import mendeliht_jl_b200 as m
from mendeliht_jl_b200 import api, bgen

import bgen_writer as bw

UKB_SAMPLE = """ID_1 ID_2 missing sex
0 0 0 D
1000017 1000017 0 1
1000023 1000023 0 2
1000035 1000035 0 2
1000041 1000041 0 1
"""


def _sample_file(tmp_path, ids, name="x.sample"):
    path = str(tmp_path / name)
    with open(path, "w") as f:
        f.write("ID_1 ID_2 missing\n0 0 0\n")
        for s in ids:
            f.write(f"{s} {s} 0\n")
    return path


def _random_file(path, n, p, nbits, seed, **kw):
    rng = np.random.default_rng(seed)
    blocks = [bw.random_block(rng, n, nbits, phased=j % 3 == 2, missing_rate=0.1) for j in range(p)]
    bw.write(path, blocks, n, **kw)


# ---- .sample files ---------------------------------------------------------------------------------------------------
def test_read_sample_file_ukb_style(tmp_path):
    path = str(tmp_path / "ukb.sample")
    open(path, "w").write(UKB_SAMPLE + "\n")
    assert bgen.read_sample_file(path) == ["1000017", "1000023", "1000035", "1000041"]


@pytest.mark.parametrize("text,msg", [
    ("ID_2 ID_1 missing\n0 0 0\na a 0\n", "line 1"),
    ("", "line 1"),
    ("ID_1 ID_2 missing\n0 0 D\na a 0\n", "line 2"),
    ("ID_1 ID_2 missing sex\n0 0 0\na a 0 1\n", "line 2"),
    ("ID_1 ID_2 missing\n0 0 0\na a 0\nb b\n", "line 4"),
])
def test_read_sample_file_rejections(tmp_path, text, msg):
    path = str(tmp_path / "bad.sample")
    open(path, "w").write(text)
    with pytest.raises(ValueError, match=msg):
        bgen.read_sample_file(path)


def test_sample_file_must_match_the_files(tmp_path):
    path = str(tmp_path / "x.bgen")
    bw.write(path, [bw.block([0, 1, 2], [1, 0, 0], 8)], 3, sample_ids=["a", "b", "c"])
    with pytest.raises(ValueError, match="lists 2 samples, the BGEN files hold 3"):
        m.B200DenseLinAlg.from_bgen(path, sample_file=_sample_file(tmp_path, ["a", "b"]))
    with pytest.raises(ValueError, match="sample 1 is 'x'"):
        m.B200DenseLinAlg.from_bgen(path, sample_file=_sample_file(tmp_path, ["a", "x", "c"]))


# ---- the row-mapped host twin -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("nbits", [1, 3, 8, 12, 15, 16, 23, 32])
def test_twin_rows_equals_full_decode_indexed(tmp_path, nbits):
    n, p = 41, 7
    path = str(tmp_path / "x.bgen")
    _random_file(path, n, p, nbits, seed=nbits, compression=nbits % 2)
    rng = np.random.default_rng(nbits + 100)
    rows = rng.permutation(n)[:23]
    cols = [0, 2, 3, 6]
    for allele in (1, 2):
        codes, miss, bits = bgen.dosage_codes(path, allele)
        c, mi, b = bgen.dosage_codes(path, allele, rows=rows, variants=cols)
        assert np.array_equal(c, codes[rows][:, cols]) and np.array_equal(mi, miss[rows][:, cols])
        assert np.array_equal(b, bits[cols])
        with bgen.BgenFile(path) as f:
            blk = f._block(3)
        full = bgen.decode_block(blk, n, allele)
        sel = bgen.decode_block(blk, n, allele, rows=rows)
        assert np.array_equal(sel[0], full[0][rows]) and np.array_equal(sel[1], full[1][rows]) and sel[2] == nbits


def test_twin_checks_kept_samples_only():
    n = 6
    # sample 4 has ploidy 3, sample 1 has a + b = 300 > 255; samples 0, 2, 3, 5 are fine
    blk = bw.block([0, 200, 255, 0, 0, 10], [0, 100, 0, 255, 0, 20], 8, ploidy=[2, 2, 2, 2, 3, 2])
    codes, miss, _ = bgen.decode_block(blk, n, rows=[5, 0, 3, 2])
    assert codes.tolist() == [20 + 2 * 225, 510, 255, 0] and not miss.any()
    with pytest.raises(ValueError, match="file sample 4 is not diploid"):
        bgen.decode_block(blk, n, rows=[0, 4])
    with pytest.raises(ValueError, match=r"file sample 1: P\(11\) \+ P\(12\) exceeds 1"):
        bgen.decode_block(blk, n, rows=[5, 1, 0])
    two_bad = bw.block([0, 200, 200], [0, 100, 100], 8)           # file samples 1 and 2 have a + b > D
    with pytest.raises(ValueError, match="file sample 1:"):       # the lowest file index, not the first row
        bgen.decode_block(two_bad, 3, rows=[2, 1, 0])
    with pytest.raises(ValueError, match="file sample 2:"):
        bgen.decode_block(two_bad, 3, rows=[0, 2])


def test_unselected_variants_are_never_inflated(tmp_path):
    path = str(tmp_path / "x.bgen")
    n = 5
    good = bw.block([0] * n, [255] * n, 8)
    bw.write(path, [good, good, bw.block([0] * n, [0] * n, 8, k=3), good], n, compression=1)
    data = bytearray(open(path, "rb").read())
    with bgen.BgenFile(path) as f:
        pos = int(f._data_pos[1])
    data[pos + 2] ^= 0xFF                                          # variant 1: corrupt zlib data
    open(path, "wb").write(bytes(data))
    with pytest.raises(ValueError, match="corrupt zlib"):
        bgen.dosage_codes(path)
    codes, _, _ = bgen.dosage_codes(path, variants=[0, 3])
    assert codes.tolist() == [[255, 255]] * n
    with bgen.BgenFile(path) as f:
        buf, offs = f.inflate_variants(np.array([0, 3]))
        assert buf.tobytes() == good + good and offs.tolist() == [0, len(good), 2 * len(good)]


def test_variant_batches(tmp_path):
    path = str(tmp_path / "b.bgen")
    bw.write(path, [bw.block([1] * 50, [0] * 50, 8)] * 9, 50, compression=0)
    with bgen.BgenFile(path) as f:
        blen = int(f.inflated_len[0])
        got = f.variant_batches([0, 2, 3, 5, 8], 2 * blen)
        assert [b.tolist() for b in got] == [[0, 2], [3, 5], [8]]
        assert [b.tolist() for b in f.variant_batches([1, 4], 1)] == [[1], [4]]
        assert f.variant_batches([], 1 << 30) == []
        assert [b.tolist() for b in f.variant_batches(range(9), 1 << 30)] == [list(range(9))]


# ---- from_bgen argument errors: all raised before the library is touched -------------------------------------------------
@pytest.fixture
def no_device(monkeypatch):
    def refuse():
        raise AssertionError("the library was touched")
    monkeypatch.setattr(api, "load", refuse)


def _two_files(tmp_path, ids=True):
    a, b = str(tmp_path / "a.bgen"), str(tmp_path / "b.bgen")
    sid = ["s0", "s1", "s2", "s3"] if ids else None
    bw.write(a, [bw.block([0, 1, 2, 3], [1, 0, 0, 0], 8)] * 3, 4, sample_ids=sid)
    bw.write(b, [bw.block([0, 1, 2, 3], [1, 0, 0, 0], 8)] * 2, 4, sample_ids=sid,
             variants=[(f"w{j}", f"rsb{j}", "2", 50 + j, ("C", "T")) for j in range(2)])
    return [a, b]


@pytest.mark.parametrize("kw,exc,msg", [
    (dict(samples=["s1", "zz"]), ValueError, r"samples\[1\] = 'zz' is not a sample ID"),
    (dict(samples=["s1", "s2", "s1"]), ValueError, r"samples\[0\] and samples\[2\] are both 's1'"),
    (dict(samples=[0, 4]), ValueError, r"samples\[1\] = 4 is outside"),
    (dict(samples=[-1]), ValueError, r"samples\[0\] = -1 is outside"),
    (dict(samples=[3, 1, 3]), ValueError, r"samples\[0\] and samples\[2\] are both sample 3"),
    (dict(samples=[0, "s1"]), ValueError, "all sample IDs"),
    (dict(samples=[True, False]), ValueError, "all sample IDs"),
    (dict(samples="s1"), ValueError, "not one string"),
    (dict(samples=[]), m.DimensionMismatch, "sample selection is empty"),
    (dict(variants=[True] * 4), ValueError, "mask has 4 entries, the files hold 5"),
    (dict(variants=[0, 2, 2]), ValueError, "strictly increasing"),
    (dict(variants=[3, 1]), ValueError, "strictly increasing"),
    (dict(variants=[0, 5]), ValueError, r"variants\[1\] = 5 is outside"),
    (dict(variants=[0.5]), ValueError, "integer indices"),
    (dict(variants=[]), m.DimensionMismatch, "variant selection is empty"),
    (dict(variants=[False] * 5), m.DimensionMismatch, "variant selection is empty"),
    (dict(variants=lambda v: v.chrom == "22"), m.DimensionMismatch, "variant selection is empty"),
])
def test_from_bgen_selection_arguments(tmp_path, no_device, kw, exc, msg):
    with pytest.raises(exc, match=msg):
        m.B200DenseLinAlg.from_bgen(_two_files(tmp_path), **kw)


def test_ids_need_an_id_source(tmp_path, no_device):
    paths = _two_files(tmp_path, ids=False)
    with pytest.raises(ValueError, match="embed no sample IDs"):
        m.B200DenseLinAlg.from_bgen(paths, samples=["s1"])
    # a .sample file supplies them; the unknown ID is then reported against it
    sf = _sample_file(tmp_path, ["s0", "s1", "s2", "s3"])
    with pytest.raises(ValueError, match=r"samples\[1\] = 'q' is not a sample ID of .*x.sample"):
        m.B200DenseLinAlg.from_bgen(paths, samples=["s1", "q"], sample_file=sf)
    dup = _sample_file(tmp_path, ["s0", "s1", "s1", "s3"], "dup.sample")
    with pytest.raises(ValueError, match="names more than one sample"):
        m.B200DenseLinAlg.from_bgen(paths, samples=["s1"], sample_file=dup)


# ---- iht / cross_validate forward the selection only when given ----------------------------------------------------------
class _Taken(Exception):
    pass


def test_wrappers_forward_selection_only_when_given(tmp_path, monkeypatch):
    pre = str(tmp_path / "data")
    bw.write(pre + ".bgen", [bw.block([0, 1], [1, 0], 8)], 2)

    def from_bgen(*a, **k):
        raise _Taken(("bgen", a, k))

    monkeypatch.setattr(api.B200DenseLinAlg, "from_bgen", classmethod(lambda cls, *a, **k: from_bgen(*a, **k)))
    y = np.array([1.0, 2.0])
    sel = dict(samples=["b", "a"], sample_file="x.sample", variants=[0])
    for kw, want in [({}, {"standardize": True}),
                     (sel, {"standardize": True, **sel}),
                     (dict(variants=[0]), {"standardize": True, "variants": [0]}),
                     (dict(samples=None, sample_file="s.sample"), {"standardize": True, "sample_file": "s.sample"})]:
        for call in (lambda: m.iht(pre + ".bgen", 1, phenotypes=y, **kw),
                     lambda: m.cross_validate(pre + ".bgen", phenotypes=y, path=[1], **kw)):
            with pytest.raises(_Taken) as e:
                call()
            assert e.value.args[0][1] == (pre + ".bgen",) and e.value.args[0][2] == want


@pytest.mark.parametrize("kw", [dict(samples=[0]), dict(sample_file="x.sample"), dict(variants=[0])])
def test_plink_input_rejects_selection(tmp_path, monkeypatch, kw):
    pre = str(tmp_path / "data")
    open(pre + ".bed", "wb").close()

    def plink(*a, **k):
        raise AssertionError("PLINK input was loaded")

    monkeypatch.setattr(api, "_load_plink", plink)
    with pytest.raises(ValueError, match="PLINK input"):
        m.iht(pre, 3, **kw)
    with pytest.raises(ValueError, match="PLINK input"):
        m.cross_validate(pre, path=[1], **kw)
