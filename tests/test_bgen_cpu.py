"""BGEN 1.2 reading on the host (no GPU): hand-written literal blocks with their dosages written out, the numpy twin
of the device decode on writer output, header / sample / variant metadata, the multi-file rules of from_bgen, every
host-side rejection, and the BGEN dispatch of iht / cross_validate."""
import os
import struct

import numpy as np
import pytest

import mendeliht_jl_b200 as m
from mendeliht_jl_b200 import _lib, api, bgen

import bgen_writer as bw


def _hdr(n, nbits, phased=0, ploidy=None):
    pl = bytes(ploidy) if ploidy is not None else bytes([2] * n)
    return struct.pack("<IHBB", n, 2, 2, 2) + pl + bytes([phased, nbits])


# ---- literal blocks: bytes and dosages written out by hand ------------------------------------------------------------
def test_literal_b8_unphased():
    # (a, b) = (255, 0), (0, 255), (0, 0), (100, 55): dosages of the second allele 0, 1, 2, (55 + 2 * 100) / 255 = 1
    blk = _hdr(4, 8) + bytes([0xFF, 0x00, 0x00, 0xFF, 0x00, 0x00, 0x64, 0x37])
    codes, miss, b = bgen.decode_block(blk, 4, allele=2)
    assert b == 8 and not miss.any()
    assert codes.tolist() == [0, 255, 510, 255]
    assert (codes / 255).tolist() == [0.0, 1.0, 2.0, 1.0]
    codes1, _, _ = bgen.decode_block(blk, 4, allele=1)
    assert codes1.tolist() == [510, 255, 0, 255]


def test_literal_b8_phased():
    # (h1, h2) = (255, 255), (0, 0), (255, 0), (10, 20): second-allele dosage 2 - h1/255 - h2/255 = 0, 2, 1, 480/255
    blk = _hdr(4, 8, phased=1) + bytes([0xFF, 0xFF, 0x00, 0x00, 0xFF, 0x00, 0x0A, 0x14])
    codes, miss, b = bgen.decode_block(blk, 4)
    assert b == 8 and codes.tolist() == [0, 510, 255, 480]
    codes1, _, _ = bgen.decode_block(blk, 4, allele=1)
    assert codes1.tolist() == [510, 0, 255, 30]


def test_literal_b3_crosses_bytes():
    # B = 3, values 7, 0, 1, 2 LSB first: bits 111 000 100 010 -> bytes 0b01000111, 0b0100; D = 7
    # sample 0 (a, b) = (7, 0): 0;  sample 1 (1, 2): c = 4, code = 2 + 8 = 10 -> dosage 10/7
    blk = _hdr(2, 3) + bytes([0x47, 0x04])
    codes, _, b = bgen.decode_block(blk, 2)
    assert b == 3 and codes.tolist() == [0, 10]


def test_literal_missing_sample():
    # sample 1 missing (ploidy byte 0x82, values stored as zeros); sample 0 (a, b) = (0, 255): dosage 1
    blk = _hdr(2, 8, ploidy=[2, 0x82]) + bytes([0x00, 0xFF, 0x00, 0x00])
    codes, miss, _ = bgen.decode_block(blk, 2)
    assert miss.tolist() == [False, True] and codes.tolist() == [255, 0]


def test_literal_b16_and_b32():
    blk = _hdr(1, 16) + struct.pack("<HH", 1000, 2000)          # D = 65535, c = 62535, code = 2000 + 125070
    assert bgen.decode_block(blk, 1)[0].tolist() == [127070]
    blk = _hdr(1, 32, phased=1) + struct.pack("<II", 1, 2)       # 2 (2^32 - 1) - 3
    assert bgen.decode_block(blk, 1)[0].tolist() == [2 * (2 ** 32 - 1) - 3]


def test_literal_file_roundtrip(tmp_path):
    path = str(tmp_path / "lit.bgen")
    blk = _hdr(4, 8) + bytes([0xFF, 0x00, 0x00, 0xFF, 0x00, 0x00, 0x64, 0x37])
    bw.write(path, [blk, blk], 4, compression=1)
    codes, miss, bits = bgen.dosage_codes(path)
    assert codes.T.tolist() == [[0, 255, 510, 255]] * 2 and bits.tolist() == [8, 8] and not miss.any()


# ---- the host twin on writer output ------------------------------------------------------------------------------------
@pytest.mark.parametrize("nbits", [1, 3, 8, 12, 15, 16, 23, 32])
@pytest.mark.parametrize("compression", [0, 1])
def test_twin_on_writer_output(tmp_path, nbits, compression):
    rng = np.random.default_rng(nbits)
    n, p = 37, 6
    den = (1 << nbits) - 1
    blocks, want, wmiss = [], [], []
    for j in range(p):
        phased = j % 2 == 1
        v0 = rng.integers(0, den + 1, size=n, dtype=np.int64)
        v1 = rng.integers(0, den + 1, size=n, dtype=np.int64) if phased else \
            np.minimum(np.floor(rng.random(n) * (den - v0 + 1)).astype(np.int64), den - v0)
        miss = rng.random(n) < 0.1
        blocks.append(bw.block(v0, v1, nbits, phased, miss))
        c2 = 2 * den - v0 - v1 if phased else v1 + 2 * (den - v0 - v1)
        want.append(np.where(miss, 0, c2)); wmiss.append(miss)
    path = str(tmp_path / "x.bgen")
    bw.write(path, blocks, n, compression=compression, sample_ids=[f"s{i}" for i in range(n)], free_data=b"xyz",
             pad=5)
    for allele in (1, 2):
        codes, miss, bits = bgen.dosage_codes(path, allele)
        w = np.array(want).T
        w = w if allele == 2 else np.where(np.array(wmiss).T, 0, 2 * den - w)
        assert np.array_equal(codes, w) and np.array_equal(miss, np.array(wmiss).T)
        assert bits.tolist() == [nbits] * p


def test_hardcall_block_matches_plink_dosages():
    g = np.array([0.0, 1.0, 2.0, np.nan, 2.0])
    codes, miss, b = bgen.decode_block(bw.hardcall_block(g), 5)
    assert b == 8 and miss.tolist() == [False, False, False, True, False]
    assert codes.tolist() == [0, 255, 510, 0, 510]


# ---- metadata ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("compression", [0, 1])
@pytest.mark.parametrize("with_ids", [False, True])
def test_metadata(tmp_path, compression, with_ids):
    n = 3
    blk = bw.block([0, 1, 2], [1, 2, 0], 2)
    variants = [("chr1:10", "rs10", "1", 10, ("A", "C")), ("", "rs77", "X", 4_000_000_000, ("GT", "G"))]
    ids = ["a", "bb", "ccc"] if with_ids else None
    path = str(tmp_path / "m.bgen")
    bw.write(path, [blk, blk], n, variants, compression=compression, sample_ids=ids, free_data=b"free", pad=11)
    with bgen.BgenFile(path) as f:
        assert (f.n, f.m, f.layout, f.compression) == (3, 2, 2, compression)
        assert f.free_data == b"free" and f.samples == ids
        assert [(v.varid, v.rsid, v.chrom, v.pos, v.alleles) for v in f.variants] == variants
        assert f.variants[1].name() == "rs77"
        buf, offs = f.inflate(0, 2)
        assert offs.tolist() == [0, len(blk), 2 * len(blk)] and buf.tobytes() == blk + blk
        assert bgen.block_bits(buf, offs, n).tolist() == [2, 2]


def test_zero_magic_accepted(tmp_path):
    path = str(tmp_path / "z.bgen")
    bw.write(path, [bw.block([1], [0], 1)], 1, magic=b"\0\0\0\0")
    assert bgen.dosage_codes(path)[0].tolist() == [[0]]


def test_batches_cover_every_variant(tmp_path):
    path = str(tmp_path / "b.bgen")
    bw.write(path, [bw.block([1] * 50, [0] * 50, 8)] * 7, 50, compression=0)
    with bgen.BgenFile(path) as f:
        blen = int(f.inflated_len[0])
        assert f.batches(2 * blen) == [(0, 2), (2, 4), (4, 6), (6, 7)]
        assert f.batches(1) == [(c, c + 1) for c in range(7)]
        assert f.batches(1 << 30) == [(0, 7)]


# ---- host-side rejections ------------------------------------------------------------------------------------------------
def _raw_file(tmp_path, **kw):
    path = str(tmp_path / "r.bgen")
    bw.write(path, [bw.block([0, 1], [1, 0], 8)], 2, **kw)
    return path


def test_reject_layout1(tmp_path):
    with pytest.raises(ValueError, match="layout 1"):
        bgen.BgenFile(_raw_file(tmp_path, layout=1))


def test_reject_zstd(tmp_path):
    with pytest.raises(ValueError, match="zstd"):
        bgen.BgenFile(_raw_file(tmp_path, compression=2))


def test_reject_bad_magic(tmp_path):
    with pytest.raises(ValueError, match="magic"):
        bgen.BgenFile(_raw_file(tmp_path, magic=b"bgem"))


@pytest.mark.parametrize("cut", [3, 12, 30, 45, 1])
def test_reject_truncated(tmp_path, cut):
    path = _raw_file(tmp_path, compression=0)
    data = open(path, "rb").read()
    with open(path, "wb") as f:
        f.write(data[:len(data) - cut] if cut != 3 else data[:3])
    with pytest.raises(ValueError, match="truncated"):
        bgen.BgenFile(path)


def test_reject_more_variants_than_stored(tmp_path):
    with pytest.raises(ValueError, match="truncated"):
        bgen.BgenFile(_raw_file(tmp_path, m=2))


def test_reject_block_n_differs_from_header(tmp_path):
    path = str(tmp_path / "n.bgen")
    bw.write(path, [bw.block([0, 1], [1, 0], 8), bw.block([0, 1, 1], [1, 0, 0], 8)], 2)
    with bgen.BgenFile(path) as f:
        with pytest.raises(ValueError, match="rs2.*3 samples, the header 2"):
            f.inflate(0, 2)
    with pytest.raises(ValueError, match="rs2"):
        bgen.dosage_codes(path)
    with pytest.raises(ValueError, match="3 samples, the header 2"):       # raised before the device is touched
        m.B200DenseLinAlg.from_bgen(path)


def test_reject_corrupt_zlib(tmp_path):
    path = _raw_file(tmp_path, compression=1)
    data = bytearray(open(path, "rb").read())
    data[-3] ^= 0xFF
    open(path, "wb").write(bytes(data))
    with pytest.raises(ValueError, match="rs1"):
        bgen.dosage_codes(path)


@pytest.mark.parametrize("blk,msg", [
    (bw.block([0, 1], [1, 0], 8, k=3), "3 alleles"),
    (bw.block([0, 1], [1, 0], 8, ploidy=[2, 3]), "sample 1 is not diploid"),
    (bw.block([200, 1], [100, 0], 8), r"sample 0: P\(11\) \+ P\(12\) exceeds 1"),
    (bw.block([0, 1], [1, 0], 8, truncate=1), "shorter than its header"),
    (bw.block([0, 1], [1, 0], 0)[:12], "B = 0"),
    (_hdr(2, 33) + bytes(20), "B = 33"),
    (_hdr(2, 8, phased=2) + bytes(4), "phased flag 2"),
])
def test_twin_rejections(tmp_path, blk, msg):
    with pytest.raises(ValueError, match=msg):
        bgen.decode_block(blk, 2)


def test_twin_missing_sample_ignores_values_and_ploidy():
    # a missing sample's ploidy and values are not checked
    blk = _hdr(2, 8, ploidy=[0x81, 2]) + bytes([0xFF, 0xFF, 0x00, 0xFF])
    codes, miss, _ = bgen.decode_block(blk, 2)
    assert miss.tolist() == [True, False] and codes.tolist() == [0, 255]


# ---- from_bgen argument and multi-file rules (all raise before the device is used) ---------------------------------------
def test_from_bgen_arguments(tmp_path):
    path = _raw_file(tmp_path)
    with pytest.raises(ValueError, match="allele"):
        m.B200DenseLinAlg.from_bgen(path, allele=3)
    with pytest.raises(ValueError, match="storage"):
        m.B200DenseLinAlg.from_bgen(path, storage="f32")
    with pytest.raises(ValueError, match="at least one"):
        m.B200DenseLinAlg.from_bgen([])


def test_from_bgen_files_must_agree(tmp_path):
    a, b, c = (str(tmp_path / f"{s}.bgen") for s in "abc")
    bw.write(a, [bw.block([0, 1], [1, 0], 8)], 2, sample_ids=["s1", "s2"])
    bw.write(b, [bw.block([0, 1, 0], [1, 0, 0], 8)], 3)
    bw.write(c, [bw.block([0, 1], [1, 0], 8)], 2, sample_ids=["s1", "t2"])
    with pytest.raises(m.DimensionMismatch, match="3 samples"):
        m.B200DenseLinAlg.from_bgen([a, b])
    with pytest.raises(ValueError, match="sample identifiers differ"):
        m.B200DenseLinAlg.from_bgen([a, c])


# ---- iht / cross_validate dispatch ---------------------------------------------------------------------------------------
class _Taken(Exception):
    pass


def test_dispatch(tmp_path, monkeypatch):
    pre = str(tmp_path / "data")
    bw.write(pre + ".bgen", [bw.block([0, 1], [1, 0], 8)], 2)
    assert api._bgen_input(pre) == pre + ".bgen"
    assert api._bgen_input(pre + ".bgen") == pre + ".bgen"
    assert api._bgen_input(str(tmp_path / "nothing")) is None
    open(pre + ".bed", "wb").close()                      # a PLINK prefix keeps precedence
    assert api._bgen_input(pre) is None

    def plink(*a, **k):
        raise _Taken("plink")

    def from_bgen(*a, **k):
        raise _Taken(("bgen", a, k))

    monkeypatch.setattr(api, "_load_plink", plink)
    monkeypatch.setattr(api.B200DenseLinAlg, "from_bgen", classmethod(lambda cls, *a, **k: from_bgen(*a, **k)))
    with pytest.raises(_Taken, match="plink"):
        m.iht(pre, 3)
    with pytest.raises(_Taken, match="plink"):
        m.cross_validate(pre, path=[1, 2])
    y = np.array([1.0, 2.0])
    for call in (lambda: m.iht(pre + ".bgen", 1, phenotypes=y), lambda: m.cross_validate(pre + ".bgen", phenotypes=y)):
        with pytest.raises(_Taken) as e:
            call()
        assert e.value.args[0][1] == (pre + ".bgen",) and e.value.args[0][2] == {"standardize": True}


@pytest.mark.parametrize("pheno", [6, np.int64(6)])
def test_bgen_rejects_fam_column_phenotypes(tmp_path, pheno):
    path = _raw_file(tmp_path)
    with pytest.raises(ValueError, match="no .fam"):
        m.iht(path, 1, phenotypes=pheno)
    with pytest.raises(ValueError, match="no .fam"):
        m.cross_validate(path, phenotypes=pheno, path=[1])
