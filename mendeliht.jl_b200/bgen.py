"""BGEN 1.2 reader (layout 2, uncompressed or zlib): header, sample IDs, variant metadata and the inflated probability
blocks that `ihtb_geno_load_bgen_columns` decodes on the device; plus `dosage_codes`, a numpy twin of that decode.

Format subset (BGEN v1.2 specification):
  bytes 0-3            uint32 offset; the first variant block starts at byte offset + 4
  header block         uint32 LH, M, N, magic b"bgen" (or four zero bytes), LH - 20 bytes of free data, uint32 flags
                       (bits 0-1 compression 0 none / 1 zlib / 2 zstd, bits 2-5 layout, bit 31 sample IDs present)
  sample IDs (bit 31)  uint32 length, uint32 N, N x (uint16 length, bytes)
  variant (layout 2)   uint16-length varid, rsid, chromosome; uint32 position; uint16 K; K x (uint32 length, allele);
                       uint32 C; compressed: uint32 D (inflated length) + C - 4 bytes of zlib data, else C bytes
  probability block    uint32 N, uint16 K, uint8 Pmin, Pmax, N ploidy bytes (bit 7 missing), uint8 phased, uint8 B,
                       then 2 N B-bit values packed least-significant bit first
Everything else (layout 1, zstd, a bad magic, a truncated file) raises ValueError.
"""
from __future__ import annotations

import mmap
import os
import struct
import zlib
from concurrent.futures import ThreadPoolExecutor
from dataclasses import dataclass

import numpy as np

COMPRESSION_NONE, COMPRESSION_ZLIB, COMPRESSION_ZSTD = 0, 1, 2
INFLATE_BATCH_BYTES = 64 << 20        # inflated bytes handed to the device per load call


@dataclass(frozen=True)
class BgenVariant:
    varid: str
    rsid: str
    chrom: str
    pos: int
    alleles: tuple

    def name(self) -> str:
        """rsid, or varid when the rsid is empty"""
        return self.rsid or self.varid


class BgenFile:
    """The index of one BGEN file: header fields, sample IDs (or None), variants, and where each variant's
    probability data lies.  The file is memory-mapped; `inflate(c0, c1)` returns the inflated blocks of variants
    [c0, c1) as (uint8 buffer, int64 offsets[c1 - c0 + 1])."""

    def __init__(self, path: str):
        self.path = os.fspath(path)
        with open(self.path, "rb") as f:
            size = os.fstat(f.fileno()).st_size
            self._mm = mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ) if size else b""
        self._parse()

    # -- parsing ------------------------------------------------------------------------------------------------------
    def _need(self, pos: int, nbytes: int, what: str) -> None:
        if pos + nbytes > len(self._mm):
            raise ValueError(f"{self.path}: truncated file ({what} needs bytes {pos}..{pos + nbytes}, the file has "
                             f"{len(self._mm)})")

    def _u(self, fmt: str, pos: int, what: str):
        self._need(pos, struct.calcsize(fmt), what)
        return struct.unpack_from(fmt, self._mm, pos)

    def _str16(self, pos: int, what: str):
        (ln,) = self._u("<H", pos, what)
        self._need(pos + 2, ln, what)
        return bytes(self._mm[pos + 2:pos + 2 + ln]).decode("utf-8", "replace"), pos + 2 + ln

    def _parse(self) -> None:
        (offset,) = self._u("<I", 0, "the offset")
        lh, m, n = self._u("<III", 4, "the header block")
        self._need(4, lh, "the header block")
        magic = bytes(self._mm[16:20])
        if magic not in (b"bgen", b"\0\0\0\0"):
            raise ValueError(f"{self.path}: not a BGEN file (magic {magic!r})")
        if lh < 20:
            raise ValueError(f"{self.path}: header length {lh} is shorter than its fields")
        (flags,) = self._u("<I", 4 + lh - 4, "the header flags")
        self.compression = flags & 3
        self.layout = (flags >> 2) & 15
        if self.compression == COMPRESSION_ZSTD:
            raise ValueError(f"{self.path}: zstd-compressed BGEN is not supported (zlib or uncompressed only)")
        if self.compression not in (COMPRESSION_NONE, COMPRESSION_ZLIB):
            raise ValueError(f"{self.path}: unknown compression {self.compression}")
        if self.layout != 2:
            raise ValueError(f"{self.path}: BGEN layout {self.layout} is not supported (layout 2 only)")
        self.n, self.m = int(n), int(m)
        self.free_data = bytes(self._mm[20:4 + lh - 4])
        self.samples = None
        if flags >> 31:
            pos = 4 + lh
            _, ns = self._u("<II", pos, "the sample identifiers")
            if ns != n:
                raise ValueError(f"{self.path}: the sample identifier block lists {ns} samples, the header {n}")
            pos += 8
            ids = []
            for _ in range(ns):
                s, pos = self._str16(pos, "the sample identifiers")
                ids.append(s)
            self.samples = ids
        pos = offset + 4
        variants, data_pos, data_len, infl_len = [], [], [], []
        for v in range(m):
            what = f"variant {v}"
            varid, pos = self._str16(pos, what)
            rsid, pos = self._str16(pos, what)
            chrom, pos = self._str16(pos, what)
            vpos, k = self._u("<IH", pos, what)
            pos += 6
            alleles = []
            for _ in range(k):
                (ln,) = self._u("<I", pos, what)
                self._need(pos + 4, ln, what)
                alleles.append(bytes(self._mm[pos + 4:pos + 4 + ln]).decode("utf-8", "replace"))
                pos += 4 + ln
            (c,) = self._u("<I", pos, what)
            pos += 4
            if self.compression == COMPRESSION_ZLIB:
                if c < 4:
                    raise ValueError(f"{self.path}: {what} has a compressed length {c} < 4")
                (d,) = self._u("<I", pos, what)
                start, clen = pos + 4, c - 4
            else:
                d, start, clen = c, pos, c
            self._need(start, clen, what + " probability data")
            variants.append(BgenVariant(varid, rsid, chrom, int(vpos), tuple(alleles)))
            data_pos.append(start); data_len.append(clen); infl_len.append(d)
            pos = start + clen
        self.variants = variants
        self._data_pos = np.asarray(data_pos, dtype=np.int64)
        self._data_len = np.asarray(data_len, dtype=np.int64)
        self.inflated_len = np.asarray(infl_len, dtype=np.int64)

    # -- probability data ---------------------------------------------------------------------------------------------
    def _block(self, c: int) -> bytes:
        s, ln = int(self._data_pos[c]), int(self._data_len[c])
        raw = self._mm[s:s + ln]
        if self.compression == COMPRESSION_NONE:
            return bytes(raw)
        try:
            out = zlib.decompress(raw)
        except zlib.error as e:
            raise ValueError(f"{self.path}: variant {c} ({self.variants[c].name()}): corrupt zlib data: {e}") from None
        if len(out) != self.inflated_len[c]:
            raise ValueError(f"{self.path}: variant {c} ({self.variants[c].name()}) inflates to {len(out)} bytes, the "
                             f"file says {int(self.inflated_len[c])}")
        return out

    def inflate(self, c0: int, c1: int, pool: ThreadPoolExecutor = None):
        """(uint8 buffer, int64 offsets) of the inflated blocks of variants [c0, c1); zlib.decompress releases the GIL,
        so a thread pool inflates blocks in parallel.  Every block's N is checked against the header's."""
        idx = range(c0, c1)
        parts = list(pool.map(self._block, idx)) if pool is not None else [self._block(c) for c in idx]
        lens = np.fromiter((len(b) for b in parts), dtype=np.int64, count=len(parts))
        offsets = np.zeros(len(parts) + 1, dtype=np.int64)
        np.cumsum(lens, out=offsets[1:])
        buf = np.frombuffer(b"".join(parts), dtype=np.uint8) if parts else np.zeros(0, np.uint8)
        for i, b in enumerate(parts):
            if len(b) < 4:
                raise ValueError(f"{self.path}: variant {c0 + i} ({self.variants[c0 + i].name()}): probability block "
                                 f"of {len(b)} bytes is truncated")
            (bn,) = struct.unpack_from("<I", b, 0)
            if bn != self.n:
                raise ValueError(f"{self.path}: variant {c0 + i} ({self.variants[c0 + i].name()}) holds {bn} samples, "
                                 f"the header {self.n}")
        return buf, offsets

    def batches(self, target: int = INFLATE_BATCH_BYTES):
        """[(c0, c1)] runs of whole variants of about `target` inflated bytes each (at least one variant)."""
        out, c0, acc = [], 0, 0
        for c in range(self.m):
            if c > c0 and acc + self.inflated_len[c] > target:
                out.append((c0, c))
                c0, acc = c, 0
            acc += int(self.inflated_len[c])
        if self.m > c0:
            out.append((c0, self.m))
        return out

    def close(self):
        if isinstance(self._mm, mmap.mmap):
            self._mm.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def block_bits(buf: np.ndarray, offsets: np.ndarray, n: int) -> np.ndarray:
    """B of every block of an inflated batch (0 where the block is too short to hold it)."""
    pos = offsets[:-1] + 9 + n
    ok = pos < offsets[1:]
    out = np.zeros(offsets.shape[0] - 1, dtype=np.int64)
    out[ok] = buf[pos[ok]]
    return out


def decode_block(block: bytes, n: int, allele: int = 2):
    """numpy twin of k_bgen_decode for one inflated block: (int64 codes[n], bool missing[n], B), code / (2^B - 1) the
    dosage of `allele`.  Raises ValueError on everything the kernel rejects."""
    b = np.frombuffer(block, dtype=np.uint8)
    if b.shape[0] < 8:
        raise ValueError("block shorter than its header")
    bn, k = struct.unpack_from("<IH", block, 0)
    if bn != n:
        raise ValueError(f"block holds N = {bn} samples, expected {n}")
    if k != 2:
        raise ValueError(f"{k} alleles (only biallelic variants)")
    if b.shape[0] < 10 + n:
        raise ValueError("block shorter than its header")
    ploidy = b[8:8 + n]
    phased, nbits = int(b[8 + n]), int(b[9 + n])
    if phased > 1:
        raise ValueError(f"phased flag {phased} is not 0 or 1")
    if not 1 <= nbits <= 32:
        raise ValueError(f"B = {nbits} bits per probability (1..32)")
    need = 10 + n + (2 * n * nbits + 7) // 8
    if b.shape[0] < need:
        raise ValueError("block shorter than its header + ceil(2 N B / 8) bytes")
    missing = (ploidy & 0x80) != 0
    bad = ~missing & ((ploidy & 63) != 2)
    if bad.any():
        raise ValueError(f"sample {int(np.flatnonzero(bad)[0])} is not diploid (only diploid samples)")
    bits = np.unpackbits(b[10 + n:need], bitorder="little")[:2 * n * nbits].reshape(2 * n, nbits).astype(np.uint64)
    vals = bits @ (np.uint64(1) << np.arange(nbits, dtype=np.uint64))
    v0, v1 = vals[0::2].astype(np.int64), vals[1::2].astype(np.int64)
    den = (1 << nbits) - 1
    if phased:
        c2 = 2 * den - v0 - v1
    else:
        over = ~missing & (v0 + v1 > den)
        if over.any():
            raise ValueError(f"sample {int(np.flatnonzero(over)[0])}: P(11) + P(12) exceeds 1 (a + b > 2^B - 1)")
        c2 = v1 + 2 * (den - v0 - v1)
    codes = c2 if allele == 2 else 2 * den - c2
    codes = np.where(missing, 0, codes)
    return codes, missing, nbits


def dosage_codes(path: str, allele: int = 2):
    """Host twin of the device ingest, for tests and small files: (int64 codes [n, p], bool missing [n, p], int64 B [p])
    with the dosage of `allele` (1 or 2) of sample i at variant j equal to codes[i, j] / (2^B[j] - 1); missing entries
    have code 0."""
    if allele not in (1, 2):
        raise ValueError(f"allele must be 1 or 2, got {allele!r}")
    with BgenFile(path) as f:
        n, p = f.n, f.m
        codes = np.zeros((n, p), dtype=np.int64)
        missing = np.zeros((n, p), dtype=bool)
        bits = np.zeros(p, dtype=np.int64)
        for c in range(p):
            try:
                codes[:, c], missing[:, c], bits[c] = decode_block(f._block(c), n, allele)
            except ValueError as e:
                raise ValueError(f"{path}: variant {c} ({f.variants[c].name()}): {e}") from None
    return codes, missing, bits
