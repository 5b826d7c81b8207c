"""A minimal BGEN 1.2 writer (layout 2) for the tests: probability blocks from explicit B-bit values, files with or
without sample IDs, free header data, padding before the first variant, zlib or no compression.  It shares the
author's reading of the specification with mendeliht.jl_b200.bgen; the hand-written literal cases of test_bgen_cpu.py
are the independent anchor."""
import struct
import zlib

import numpy as np


def pack_values(vals, nbits: int) -> bytes:
    """B-bit values packed least-significant bit first, value i at bits [i B, (i + 1) B)"""
    v = np.asarray(vals, dtype=np.uint64)
    if nbits == 8:
        return v.astype(np.uint8).tobytes()
    bits = ((v[:, None] >> np.arange(nbits, dtype=np.uint64)) & np.uint64(1)).astype(np.uint8).reshape(-1)
    return np.packbits(bits, bitorder="little").tobytes()


def block(v0, v1, nbits: int, phased: bool = False, missing=None, ploidy=None, k: int = 2, n: int = None,
          truncate: int = 0) -> bytes:
    """One inflated probability block: per sample i the values (v0[i], v1[i]) -- (P(11), P(12)) unphased, (h1, h2)
    phased; `missing` marks samples (their values are written as zeros), `ploidy` overrides the ploidy bytes."""
    v0 = np.asarray(v0, dtype=np.uint64)
    v1 = np.asarray(v1, dtype=np.uint64)
    nn = v0.shape[0]
    miss = np.zeros(nn, dtype=bool) if missing is None else np.asarray(missing, dtype=bool)
    pl = np.full(nn, 2, dtype=np.uint8) if ploidy is None else np.asarray(ploidy, dtype=np.uint8)
    pl = pl | (miss.astype(np.uint8) << 7)
    vals = np.empty(2 * nn, dtype=np.uint64)
    vals[0::2] = np.where(miss, 0, v0)
    vals[1::2] = np.where(miss, 0, v1)
    out = struct.pack("<IHBB", nn if n is None else n, k, 2, 2) + pl.tobytes() + struct.pack("<BB", int(phased), nbits)
    out += pack_values(vals, nbits)
    return out[:len(out) - truncate] if truncate else out


def random_block(rng, n: int, nbits: int, phased: bool = False, missing_rate: float = 0.0) -> bytes:
    """Random valid probabilities on the grid 1 / (2^B - 1), including the corners 0 and D."""
    den = (1 << nbits) - 1
    if phased:
        v0 = rng.integers(0, den + 1, size=n, dtype=np.int64)
        v1 = rng.integers(0, den + 1, size=n, dtype=np.int64)
    else:
        v0 = rng.integers(0, den + 1, size=n, dtype=np.int64)
        v1 = np.floor(rng.random(n) * (den - v0 + 1)).astype(np.int64)
        v1 = np.minimum(v1, den - v0)
        corner = rng.random(n) < 0.2                       # hard calls: (D, 0), (0, D), (0, 0)
        pick = rng.integers(0, 3, size=n)
        v0 = np.where(corner, np.where(pick == 0, den, 0), v0)
        v1 = np.where(corner, np.where(pick == 1, den, 0), v1)
    miss = rng.random(n) < missing_rate if missing_rate else None
    return block(v0, v1, nbits, phased, miss)


def hardcall_block(dosage, nbits: int = 8) -> bytes:
    """Hard calls: dosage of the second allele 0 / 1 / 2, NaN missing -> unphased probabilities (D, 0) / (0, D) /
    (0, 0)."""
    g = np.asarray(dosage, dtype=np.float64)
    den = (1 << nbits) - 1
    miss = np.isnan(g)
    v0 = np.where(g == 0, den, 0)
    v1 = np.where(g == 1, den, 0)
    return block(v0, v1, nbits, False, miss)


def _s16(s: str) -> bytes:
    b = s.encode()
    return struct.pack("<H", len(b)) + b


def write(path, blocks, n: int, variants=None, compression: int = 1, sample_ids=None, free_data: bytes = b"",
          pad: int = 0, layout: int = 2, magic: bytes = b"bgen", m: int = None, level: int = 6) -> None:
    """A BGEN file of the inflated `blocks`.  variants: [(varid, rsid, chrom, pos, alleles)] (default rs<j>, chr 1)."""
    if variants is None:
        variants = [(f"v{j}", f"rs{j + 1}", "1", 1000 + j, ("A", "G")) for j in range(len(blocks))]
    flags = compression | (layout << 2) | ((1 << 31) if sample_ids is not None else 0)
    lh = 20 + len(free_data)
    header = struct.pack("<III", lh, len(blocks) if m is None else m, n) + magic + free_data + struct.pack("<I", flags)
    samples = b""
    if sample_ids is not None:
        body = b"".join(_s16(s) for s in sample_ids)
        samples = struct.pack("<II", 8 + len(body), len(sample_ids)) + body
    offset = len(header) + len(samples) + pad
    out = [struct.pack("<I", offset), header, samples, b"\0" * pad]
    for (varid, rsid, chrom, pos, alleles), blk in zip(variants, blocks):
        meta = _s16(varid) + _s16(rsid) + _s16(chrom) + struct.pack("<IH", pos, len(alleles))
        meta += b"".join(struct.pack("<I", len(a.encode())) + a.encode() for a in alleles)
        if compression == 1:
            z = zlib.compress(blk, level)
            meta += struct.pack("<II", len(z) + 4, len(blk)) + z
        else:
            meta += struct.pack("<I", len(blk)) + blk
        out.append(meta)
    with open(path, "wb") as f:
        f.write(b"".join(out))
