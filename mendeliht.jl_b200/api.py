"""Host-side mirror of MendelIHT.jl's public API over libihtb200.so.

Same names, argument meaning and error behaviour as the reference (all paths under /root/reference):
  `B200SnpLinAlg`  <- `SnpLinAlg{Float64}(s; model=ADDITIVE_MODEL, center, scale, impute)`  src/wrapper.jl:68-69
  `B200DenseLinAlg` <- a dense `x::AbstractMatrix{T}`, T = Float64 / Float32  src/fit.jl:62 (standardize_genotypes!,
                       src/wrapper.jl:406-423, on the device when asked)
                       `from_bgen` <- the dense dosages `parse_genotypes` reads from .bgen  src/wrapper.jl:451-485
  `fit_iht`        <- src/fit.jl:60-118        `IHTResult` <- src/data_structures.jl:245-258
  `cv_iht`         <- src/cross_validation.jl:60-131
  `iht`            <- src/wrapper.jl:52-120    `cross_validate` <- src/wrapper.jl:301-349  (PLINK or .bgen input)
Julia is not available in this image, so this Python layer plays the role of julia/MendelIHTB200.jl (which binds
the very same C entry points with ccall); every numerical step happens inside the CUDA library.
"""
from __future__ import annotations

import ctypes as C
import os
from concurrent.futures import ThreadPoolExecutor
from dataclasses import dataclass, field

import numpy as np

from . import _lib
from ._lib import Cfg, IterTrace, Result, check, f64, load, ptr

NORMAL, BERNOULLI, POISSON, NEGBIN = "Normal", "Bernoulli", "Poisson", "NegativeBinomial"
DIST_ID = {NORMAL: 0, BERNOULLI: 1, POISSON: 2, NEGBIN: 3}
EST_R_ID = {"None": 0, "MM": 1, "Newton": 2}
LINK_ID = {"IdentityLink": 0, "LogitLink": 1, "LogLink": 2, "ProbitLink": 3, "CloglogLink": 4, "CauchitLink": 5,
           "SqrtLink": 6, "InverseLink": 7, "InverseSquareLink": 8}


def canonicallink(d: str) -> str:
    """`canonicallink(d())`, LogLink for NegativeBinomial (src/wrapper.jl:87)."""
    return {NORMAL: "IdentityLink", BERNOULLI: "LogitLink", POISSON: "LogLink", NEGBIN: "LogLink"}[d]


class B200SnpLinAlg:
    """Device-resident 2-bit genotype matrix with SnpLinAlg semantics (n samples x p SNPs)."""

    def __init__(self, handle, n, p, j0=0):
        self._h = handle
        self.n, self.p, self.j0 = int(n), int(p), int(j0)
        self.center = self.scale = self.impute = True

    @classmethod
    def from_bed_columns(cls, bed_cols: np.ndarray, n: int, center=True, scale=True, impute=True):
        """bed_cols: uint8 [p, stride>=ceil(n/4)] SNP-major packed columns (PLINK .bed without the 3 magic bytes)."""
        bed_cols = np.ascontiguousarray(bed_cols, dtype=np.uint8)
        if bed_cols.ndim != 2:
            raise _lib.DimensionMismatch(_lib.IHTB_EDIM, "bed_cols must be [p, ceil(n/4)]")
        h = C.c_void_p()
        check(load().ihtb_geno_create(ptr(bed_cols, C.c_uint8), n, bed_cols.shape[0], bed_cols.shape[1],
                                      int(center), int(scale), int(impute), C.byref(h)))
        obj = cls(h, n, bed_cols.shape[0])
        obj.center, obj.scale, obj.impute = bool(center), bool(scale), bool(impute)
        return obj

    @classmethod
    def from_bed_file(cls, path: str, n: int, **kw):
        """One SNP-major PLINK .bed file.  The file is memory-mapped and streamed to the device in 64 MiB chunks, so
        host memory stays bounded for files larger than RAM."""
        return cls.from_bed_files([path], n, **kw)

    @classmethod
    def from_bed_files(cls, paths, n: int, center=True, scale=True, impute=True):
        """Several .bed files over the same n samples (e.g. one per chromosome), concatenated SNP-wise in the order
        given (ihtb_geno_create_empty / ihtb_geno_load_columns / ihtb_geno_finalize)."""
        stride = (n + 3) // 4
        maps = []
        for path in paths:
            mm = np.memmap(path, dtype=np.uint8, mode="r")
            if mm.shape[0] < 3 or bytes(mm[:3]) != bytes([0x6C, 0x1B, 0x01]):
                raise ValueError(f"{path}: not a SNP-major PLINK .bed file")
            if (mm.shape[0] - 3) % stride:
                raise _lib.DimensionMismatch(_lib.IHTB_EDIM, f"{path}: size is not 3 + p*ceil(n/4) bytes for n={n}")
            maps.append(mm)
        p = sum((mm.shape[0] - 3) // stride for mm in maps)
        lib = load()
        h = C.c_void_p()
        check(lib.ihtb_geno_create_empty(n, p, int(center), int(scale), int(impute), C.byref(h)))
        obj = cls(h, n, p)
        obj.center, obj.scale, obj.impute = bool(center), bool(scale), bool(impute)
        j = 0
        for mm in maps:
            cols = (mm.shape[0] - 3) // stride
            base = mm.ctypes.data + 3
            check(lib.ihtb_geno_load_columns(h, C.cast(C.c_void_p(base), C.POINTER(C.c_uint8)), stride, j, cols))
            j += cols
        check(lib.ihtb_geno_finalize(h))
        return obj

    @classmethod
    def synthetic(cls, n: int, p: int, seed: int, missing_rate: float = 0.0, j0: int = 0):
        h = C.c_void_p()
        check(load().ihtb_geno_create_synthetic(n, p, j0, seed, missing_rate, C.byref(h)))
        return cls(h, n, p, j0)

    @property
    def shape(self):
        return (self.n, self.p)

    def ternary_tiles(self) -> np.ndarray:
        """Raw bytes of the ternary copy the FAST / PAIR sweeps stream (format: include/ihtb200.h, synth.ternary_tiles)."""
        nbytes, tern = self.sweep_stream_bytes()
        if not tern:
            raise _lib.IHTBError(_lib.IHTB_EINVAL, "this handle holds no ternary copy")
        out = np.empty(nbytes, dtype=np.uint8)
        check(load().ihtb_geno_ternary_tiles(self._h, ptr(out, C.c_uint8), nbytes))
        return out

    def gather_bench(self, ncols: int, reps: int = 5):
        """(ms per exact re-scoring of `ncols` columns, max difference to the per-column kernel / max |value|)"""
        ms, err = C.c_double(0.0), C.c_double(0.0)
        check(load().ihtb_gather_bench(self._h, int(ncols), int(reps), C.byref(ms), C.byref(err)))
        return float(ms.value), float(err.value)

    def sweep_stream_bytes(self):
        """(bytes of packed genotypes one FAST / PAIR sweep reads from HBM, ternary copy in use?)"""
        b, t = C.c_int64(0), C.c_int32(0)
        check(load().ihtb_geno_sweep_stream_bytes(self._h, C.byref(b), C.byref(t)))
        return int(b.value), bool(t.value)

    def size(self, dim=None):
        return self.shape if dim is None else self.shape[dim - 1]

    def stats(self):
        mu = np.empty(self.p); sinv = np.empty(self.p); nm = np.empty(self.p, dtype=np.int64)
        check(load().ihtb_geno_stats(self._h, ptr(mu, C.c_double), ptr(sinv, C.c_double), ptr(nm, C.c_int64)))
        return mu, sinv, nm

    def counts(self) -> np.ndarray:
        """SnpArrays `counts(s, dims=1)`: int64 [4, p], rows = codes 00, 01 (missing), 10, 11."""
        out = np.empty((self.p, 4), dtype=np.int64)
        check(load().ihtb_geno_counts(self._h, ptr(out, C.c_int64)))
        return out.T

    def maf(self) -> np.ndarray:
        """SnpArrays `maf(s)`: minor allele frequency of every SNP."""
        out = np.empty(self.p)
        check(load().ihtb_geno_maf(self._h, ptr(out, C.c_double)))
        return out

    def decode(self, i0=0, i1=None, j0=0, j1=None) -> np.ndarray:
        """x[i0:i1, j0:j1] through the getindex formula, float64 [i1-i0, j1-j0]."""
        i1 = self.n if i1 is None else i1
        j1 = self.p if j1 is None else j1
        out = np.empty((max(j1 - j0, 0), max(i1 - i0, 0)))
        check(load().ihtb_geno_decode(self._h, i0, i1, j0, j1, ptr(out, C.c_double)))
        return out.T

    def packed(self, j0=0, j1=None) -> np.ndarray:
        j1 = self.p if j1 is None else j1
        out = np.empty((max(j1 - j0, 0), (self.n + 3) // 4), dtype=np.uint8)
        check(load().ihtb_geno_packed(self._h, j0, j1, ptr(out, C.c_uint8)))
        return out

    def xt_v(self, v: np.ndarray, mode: int = _lib.SWEEP_FAST) -> np.ndarray:
        """mul!(out, Transpose(x), v) for v [n] or [n, m]."""
        v = np.asarray(v, dtype=np.float64)
        one = v.ndim == 1
        vm = np.asfortranarray(v.reshape(self.n, -1))
        if vm.shape[0] != self.n:
            raise _lib.DimensionMismatch(_lib.IHTB_EDIM, "length(v) != size(x, 1)")
        m = vm.shape[1]
        out = np.empty((self.p, m), order="F")
        check(load().ihtb_xt_v(self._h, vm.ctypes.data_as(C.POINTER(C.c_double)), m,
                               out.ctypes.data_as(C.POINTER(C.c_double)), mode))
        return out[:, 0].copy() if one else out

    def x_support(self, idx, coef) -> np.ndarray:
        """x[:, idx] * coef for coef [k] or [k, m]."""
        idx = np.ascontiguousarray(idx, dtype=np.int64)
        coef = np.asarray(coef, dtype=np.float64)
        one = coef.ndim == 1
        m = 1 if one else coef.shape[1]
        cm = np.asfortranarray(coef.reshape(idx.shape[0], m))
        out = np.empty((self.n, m), order="F")
        check(load().ihtb_x_support(self._h, ptr(idx, C.c_int64), idx.shape[0],
                                    cm.ctypes.data_as(C.POINTER(C.c_double)), m,
                                    out.ctypes.data_as(C.POINTER(C.c_double))))
        return out[:, 0].copy() if one else out

    def close(self):
        if getattr(self, "_h", None):
            load().ihtb_geno_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class B200DenseLinAlg:
    """Device-resident dense n x p design matrix (float64 or float32 entries, or 16-bit fixed-point dosage codes from
    `from_dosages`; computed on in FP64): imputed dosages from
    VCF / BGEN or any real predictors.  Works wherever a single-GPU `B200SnpLinAlg` does in `fit_iht`, `cv_iht`, `cv_run`
    and `IHTVariable` (univariate traits)."""

    # host memory of the column-block upload of a C-ordered array (one block at a time)
    _BLOCK_BYTES = 64 << 20

    def __init__(self, handle, n, p, dtype, standardize, denominator=None):
        self._h = handle
        self.n, self.p = int(n), int(p)
        self.dtype = np.dtype(dtype)
        self.standardize = bool(standardize)
        self.denominator = denominator

    @classmethod
    def from_array(cls, x: np.ndarray, standardize: bool = False) -> "B200DenseLinAlg":
        """x: float64 or float32 ndarray [n, p].  standardize=True applies `standardize_genotypes!` on the device (NaN =
        missing, imputed with the column mean; x = (g - mu) / sqrt(mu (1 - mu/2))); otherwise x is used as given and must
        be finite.  A Fortran-ordered array (or column-major view) is read in place; any other layout is uploaded in
        column blocks, so host memory grows by one block rather than by a transposed copy."""
        if not isinstance(x, np.ndarray):
            raise TypeError("x must be a numpy ndarray")
        if x.ndim != 2:
            raise _lib.DimensionMismatch(_lib.IHTB_EDIM, f"x must be a matrix (ndim 2), got ndim {x.ndim}")
        if x.dtype == np.float64:
            code = _lib.DENSE_F64
        elif x.dtype == np.float32:
            code = _lib.DENSE_F32
        else:
            raise TypeError(f"x must be float64 or float32, got {x.dtype}")
        n, p = x.shape
        if n == 0 or p == 0:
            raise _lib.DimensionMismatch(_lib.IHTB_EDIM, f"x must have n > 0 and p > 0, got {x.shape}")
        es = x.itemsize
        lib = load()
        h = C.c_void_p()
        s0, s1 = x.strides
        if s0 == es and s1 > 0 and s1 % es == 0 and s1 // es >= n:
            check(lib.ihtb_geno_create_dense(C.c_void_p(x.ctypes.data), code, n, p, s1 // es, int(bool(standardize)),
                                             C.byref(h)))
            return cls(h, n, p, x.dtype, standardize)
        check(lib.ihtb_geno_create_dense_empty(n, p, code, int(bool(standardize)), C.byref(h)))
        obj = cls(h, n, p, x.dtype, standardize)
        cols = max(1, cls._BLOCK_BYTES // (n * es))
        for j in range(0, p, cols):
            blk = np.asfortranarray(x[:, j:j + cols])
            check(lib.ihtb_geno_load_dense_columns(h, C.c_void_p(blk.ctypes.data), n, j, blk.shape[1]))
        check(lib.ihtb_geno_finalize(h))
        return obj

    @staticmethod
    def encode_dosages(x: np.ndarray, denominator: int, standardize: bool = False) -> np.ndarray:
        """The uint16 codes c = rint(x * D) of a float64 block, checked to be exact: every non-NaN entry must satisfy
        0 <= c <= 65534 and c / D == x; NaN becomes the missing code 65535 when standardizing.  Raises ValueError
        naming the first offending (i, j) (column-major order) and its value, IHTBError(IHTB_EDOMAIN) for NaN without
        standardization."""
        miss = np.isnan(x)
        if miss.any() and not standardize:
            i, j = _first_true(miss)
            raise _lib.IHTBError(_lib.IHTB_EDOMAIN, f"x[{i}, {j}] is NaN: missing dosages need standardize=True")
        xs = np.where(miss, 0.0, x)
        with np.errstate(invalid="ignore", over="ignore"):
            c = np.rint(xs * denominator)
            bad = ~((c >= 0) & (c <= 65534))
            c = np.where(bad, 0.0, c)
            bad |= c / denominator != xs
        if bad.any():
            i, j = _first_true(bad)
            raise ValueError(f"x[{i}, {j}] = {float(x[i, j])!r} is not a dosage c / {denominator} with an integer "
                             f"0 <= c <= 65534")
        codes = c.astype(np.uint16)
        codes[miss] = _lib.DOSAGE16_MISSING
        return codes

    @classmethod
    def from_dosages(cls, x: np.ndarray, denominator: int, standardize: bool = False) -> "B200DenseLinAlg":
        """Lossless 16-bit fixed-point storage of dosages that lie on the grid 1 / denominator (PLINK 2: 16384, VCF DS
        printed with d decimals: 10**d, BGEN 8-bit: 255; 1 <= denominator <= 65534).  x: float64 ndarray [n, p] in any
        layout, encoded on the host in column blocks as code c = rint(x * D) (every entry is checked: c / D == x
        exactly).  NaN is missing with standardize=True and an IHTBError(IHTB_EDOMAIN) otherwise, as in `from_array`.
        The device holds 2 bytes per entry, and every result (decode, stats, fits, cross-validation) is that of
        `from_array(x, standardize)` bit for bit; the X'v sweep reads the codes and differs only in the last bits,
        within its selection bound.  `dtype` is uint16."""
        if not isinstance(x, np.ndarray):
            raise TypeError("x must be a numpy ndarray")
        if x.ndim != 2:
            raise _lib.DimensionMismatch(_lib.IHTB_EDIM, f"x must be a matrix (ndim 2), got ndim {x.ndim}")
        if x.dtype != np.float64:
            raise TypeError(f"x must be float64, got {x.dtype}")
        if isinstance(denominator, (bool, np.bool_)) or not isinstance(denominator, (int, np.integer)):
            raise TypeError(f"denominator must be an integer, got {type(denominator).__name__}")
        denominator = int(denominator)
        if not 1 <= denominator <= 65534:
            raise ValueError(f"denominator must be in [1, 65534], got {denominator}")
        n, p = x.shape
        if n == 0 or p == 0:
            raise _lib.DimensionMismatch(_lib.IHTB_EDIM, f"x must have n > 0 and p > 0, got {x.shape}")
        cols = max(1, cls._BLOCK_BYTES // (n * 8))
        # the first block is checked before the device is touched (all of a matrix up to 64 MB); a bad entry in a later
        # block raises before that block is uploaded, and the handle is released with `obj`
        first = cls.encode_dosages(x[:, :cols], denominator, standardize)
        lib = load()
        h = C.c_void_p()
        check(lib.ihtb_geno_create_dosage16_empty(n, p, denominator, int(bool(standardize)), C.byref(h)))
        obj = cls(h, n, p, np.uint16, standardize, denominator)
        for j in range(0, p, cols):
            blk = first if j == 0 else cls.encode_dosages(x[:, j:j + cols], denominator, standardize)
            blk = np.asfortranarray(blk)
            check(lib.ihtb_geno_load_dense_columns(h, C.c_void_p(blk.ctypes.data), n, j, blk.shape[1]))
        check(lib.ihtb_geno_finalize(h))
        return obj

    @classmethod
    def from_bgen(cls, paths, standardize: bool = False, allele: int = 2, storage: str = "auto") -> "B200DenseLinAlg":
        """Dosages of BGEN 1.2 files (layout 2, uncompressed or zlib; biallelic diploid variants).  `paths`: one file or
        a list (e.g. one per chromosome) over the same samples -- N must match, and so must the sample IDs where files
        carry them -- whose variants become the columns in the order given.  A probability stored as a B-bit integer
        makes the dosage of `allele` (2, the default: copies of the second allele, what a PLINK handle counts; or 1)
        exactly code / (2^B - 1); the host inflates the blocks (thread pool, ~64 MB batches) and the device decodes them
        (ihtb_geno_load_bgen_columns).  storage="auto": 16-bit codes with denominator 2^B - 1 (as `from_dosages`) when
        the first variant has B <= 15, Float64 otherwise; "fix16" / "f64" force one (a FIX16 handle needs the same B in
        every variant).  Missing samples need standardize=True, as NaN does for `from_array`.  The handle equals
        `from_dosages(codes / D, D, standardize)` (FIX16) or `from_array(codes / D, standardize)` bit for bit
        (bgen.dosage_codes is the host twin), and carries `.variants` (bgen.BgenVariant per column) and `.samples`
        (sample IDs, or None when no file stores them)."""
        from . import bgen as _bgen
        if isinstance(paths, (str, bytes, os.PathLike)):
            paths = [paths]
        paths = [os.fspath(q) for q in paths]
        if not paths:
            raise ValueError("from_bgen needs at least one file")
        if isinstance(allele, (bool, np.bool_)) or allele not in (1, 2):
            raise ValueError(f"allele must be 1 or 2, got {allele!r}")
        if storage not in ("auto", "fix16", "f64"):
            raise ValueError(f"storage must be 'auto', 'fix16' or 'f64', got {storage!r}")
        files = []
        try:
            for q in paths:
                files.append(_bgen.BgenFile(q))
            n = files[0].n
            samples, samples_from = None, None
            for f in files:
                if f.n != n:
                    raise _lib.DimensionMismatch(_lib.IHTB_EDIM, f"{f.path} holds {f.n} samples, {files[0].path} {n}")
                if f.samples is not None:
                    if samples is None:
                        samples, samples_from = f.samples, f.path
                    elif f.samples != samples:
                        raise ValueError(f"{f.path}: sample identifiers differ from those of {samples_from}")
            p = sum(f.m for f in files)
            if n == 0 or p == 0:
                raise _lib.DimensionMismatch(_lib.IHTB_EDIM, f"BGEN input must have n > 0 samples and p > 0 variants, "
                                                             f"got n = {n}, p = {p}")
            variants = [v for f in files for v in f.variants]
            jobs, j = [], 0
            for f in files:
                for c0, c1 in f.batches(_bgen.INFLATE_BATCH_BYTES):
                    jobs.append((f, c0, c1, j + c0))
                j += f.m
            return cls._load_bgen(jobs, n, p, variants, samples, standardize, allele, storage)
        finally:
            for f in files:
                f.close()

    @classmethod
    def _load_bgen(cls, jobs, n, p, variants, samples, standardize, allele, storage):
        from . import bgen as _bgen
        lib = load()
        obj = None
        with ThreadPoolExecutor(max_workers=max(1, min(32, os.cpu_count() or 1))) as pool, \
                ThreadPoolExecutor(max_workers=1) as ahead:
            def inflate(job):
                f, c0, c1, _ = job
                return f.inflate(c0, c1, pool)
            nxt = ahead.submit(inflate, jobs[0])
            for t, job in enumerate(jobs):
                buf, offs = nxt.result()
                if t + 1 < len(jobs):
                    nxt = ahead.submit(inflate, jobs[t + 1])       # inflate the next batch while this one loads
                f, c0, c1, jcol = job
                bits = _bgen.block_bits(buf, offs, n)
                if obj is None:
                    b0 = int(bits[0])
                    if storage == "fix16" and not 1 <= b0 <= 15:
                        raise ValueError(f"{f.path}: variant {variants[0].name()} stores B = {b0} bits per probability; "
                                         f"16-bit codes need B <= 15 (use storage='f64')")
                    h = C.c_void_p()
                    if storage == "fix16" or (storage == "auto" and 1 <= b0 <= 15):
                        den = (1 << b0) - 1
                        check(lib.ihtb_geno_create_dosage16_empty(n, p, den, int(bool(standardize)), C.byref(h)))
                        obj = cls(h, n, p, np.uint16, standardize, den)
                    else:
                        check(lib.ihtb_geno_create_dense_empty(n, p, _lib.DENSE_F64, int(bool(standardize)), C.byref(h)))
                        obj = cls(h, n, p, np.float64, standardize)
                    obj.variants, obj.samples = variants, samples
                if obj.denominator is not None:
                    other = np.flatnonzero(bits != b0)
                    if other.size:
                        c = c0 + int(other[0])
                        raise ValueError(f"{f.path}: variant {f.variants[c].name()} stores B = {int(bits[other[0]])} "
                                         f"bits per probability, the first variant B = {b0}: 16-bit codes need one B "
                                         f"for all variants (use storage='f64')")
                status = lib.ihtb_geno_load_bgen_columns(obj._h, _lib.ptr(buf, C.c_uint8), _lib.ptr(offs, C.c_int64),
                                                         jcol, c1 - c0, int(allele))
                if status != _lib.IHTB_OK:
                    raise _lib._EXC.get(status, _lib.IHTBError)(status, f"{f.path}: {_lib.last_error()}")
        check(lib.ihtb_geno_finalize(obj._h))
        return obj

    @property
    def shape(self):
        return (self.n, self.p)

    def size(self, dim=None):
        return self.shape if dim is None else self.shape[dim - 1]

    def stats(self):
        """(mu, sigma_inv, n_missing) that standardization applied; (0, 1, 0) for a matrix used as given."""
        return B200SnpLinAlg.stats(self)

    def decode(self, i0=0, i1=None, j0=0, j1=None) -> np.ndarray:
        """x[i0:i1, j0:j1] as stored on the device, float64."""
        return B200SnpLinAlg.decode(self, i0, i1, j0, j1)

    def xt_v(self, v: np.ndarray, mode: int = _lib.SWEEP_FAST) -> np.ndarray:
        """x' v in FP64 for v [n] or [n, m] (every mode computes the same product)."""
        return B200SnpLinAlg.xt_v(self, v, mode)

    def x_support(self, idx, coef) -> np.ndarray:
        """x[:, idx] * coef for coef [k] or [k, m], columns added in the order given."""
        return B200SnpLinAlg.x_support(self, idx, coef)

    def sweep_stream_bytes(self):
        """(bytes one X'v sweep reads from HBM = n p sizeof(T), 2 n p for dosage codes, False)"""
        return B200SnpLinAlg.sweep_stream_bytes(self)

    def close(self):
        if getattr(self, "_h", None):
            load().ihtb_geno_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _first_true(mask: np.ndarray):
    """(i, j) of the first True entry of a 2-D mask in column-major order"""
    j = int(np.flatnonzero(mask.any(axis=0))[0])
    return int(np.flatnonzero(mask[:, j])[0]), j


class B200MultiSnpLinAlg:
    """The genotype operator over several GPUs driven by THIS process (`ihtb_mgeno`, SURVEY.md 8b `ngpu`).
    mode SHARD: SNP columns block-partitioned over the devices, `fit_iht` runs one fit over all of them;
    mode REPLICATE: the whole matrix on every device, `cv_iht` farms its (fold, k) grid over them."""
    SHARD, REPLICATE = 0, 1

    def __init__(self, handle, n, p, ngpu, mode):
        self._h = handle
        self.n, self.p, self.ngpu, self.mode = int(n), int(p), int(ngpu), int(mode)
        self.center = self.scale = self.impute = True

    @staticmethod
    def _devs(devices):
        if devices is None:
            return None
        return (C.c_int32 * len(devices))(*[int(d) for d in devices])

    @classmethod
    def from_bed_columns(cls, bed_cols: np.ndarray, n: int, ngpu: int, mode: int = 0, devices=None, center=True,
                         scale=True, impute=True):
        bed_cols = np.ascontiguousarray(bed_cols, dtype=np.uint8)
        if bed_cols.ndim != 2:
            raise _lib.DimensionMismatch(_lib.IHTB_EDIM, "bed_cols must be [p, ceil(n/4)]")
        h = C.c_void_p()
        check(load().ihtb_mgeno_create(ptr(bed_cols, C.c_uint8), n, bed_cols.shape[0], bed_cols.shape[1], int(center),
                                       int(scale), int(impute), int(ngpu), cls._devs(devices), int(mode), C.byref(h)))
        return cls(h, n, bed_cols.shape[0], ngpu, mode)

    @classmethod
    def synthetic(cls, n: int, p: int, seed: int, missing_rate: float = 0.0, ngpu: int = 2, mode: int = 0, devices=None):
        h = C.c_void_p()
        check(load().ihtb_mgeno_create_synthetic(n, p, seed, missing_rate, int(ngpu), cls._devs(devices), int(mode),
                                                 C.byref(h)))
        return cls(h, n, p, ngpu, mode)

    @property
    def shape(self):
        return (self.n, self.p)

    def part(self, i: int) -> "B200SnpLinAlg":
        """Borrowed single-device operator of part i (do not close it)."""
        h = C.c_void_p(); dev = C.c_int32(0); j0 = C.c_int64(0)
        check(load().ihtb_mgeno_part(self._h, int(i), C.byref(h), C.byref(dev), C.byref(j0)))
        n, p = C.c_int64(0), C.c_int64(0)
        check(load().ihtb_geno_dims(h, C.byref(n), C.byref(p)))
        part = B200SnpLinAlg(h, n.value, p.value, j0.value)
        part.close = lambda: None          # owned by the multi-device handle
        part.device = int(dev.value)
        return part

    def close(self):
        if getattr(self, "_h", None):
            load().ihtb_mgeno_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class SparseCoef:
    """The k non-zero coefficients of a fit as (global column, value) pairs; `dense()` is the length-p vector."""

    def __init__(self, p: int, idx: np.ndarray, val: np.ndarray):
        self.p, self.idx, self.val = int(p), idx, val

    def dense(self) -> np.ndarray:
        b = np.zeros(self.p)
        b[self.idx] = self.val
        return b


@dataclass
class IHTResult:
    """`IHTResult` (src/data_structures.jl:245-258) + device-side counters.  `beta` is the dense length-p vector of the
    reference; when the fit hands over a `SparseCoef` it is built on first access (zeroing p doubles per fit costs 5 ms at
    p = 4M -- more than a tenth of an 8-GPU fit) and `beta_sparse` keeps the pairs."""
    time: float
    logl: float
    iter: int
    beta: np.ndarray
    c: np.ndarray
    J: int
    k: int
    group: list
    d: str
    sigma_g: float
    trace: list = field(default_factory=list)   # [(logl, backtracks, tol, eta, n_candidates)] per iteration
    n_sweeps: int = 0
    n_backtracks: int = 0
    sweep_seconds: float = 0.0
    n_launches: int = 0

    def __post_init__(self):
        sp = self.__dict__.get("beta")
        if isinstance(sp, SparseCoef):
            self.__dict__["beta_sparse"] = sp
            del self.__dict__["beta"]                    # __getattr__ below builds the dense vector on first use
        else:
            self.__dict__["beta_sparse"] = None

    def __getattr__(self, name):
        if name == "beta":
            sp = self.__dict__.get("beta_sparse")
            if sp is not None:
                dense = sp.dense()
                self.__dict__["beta"] = dense
                return dense
        raise AttributeError(name)


class IHTVariable:
    """`IHTVariable` (src/data_structures.jl:4-43): one fit's device workspace."""

    def __init__(self, x: B200SnpLinAlg, z, y, k, d=NORMAL, l="IdentityLink", zkeep=None, nb_r=1.0, tol=1e-4,
                 max_iter=200, min_iter=5, max_step=3, sweep_mode=_lib.SWEEP_FAST, comm=None, p_global=None,
                 est_r="None", weight=None, debias=False, J=1, group=None):
        y = f64(y)
        z = np.asarray(z, dtype=np.float64)
        if z.ndim == 1:
            z = z.reshape(-1, 1)
        n = x.n
        if not (y.shape[0] == n == z.shape[0]):
            raise _lib.DimensionMismatch(
                _lib.IHTB_EDIM, f"row dimension of y, x, and z ({y.shape[0]}, {n}, {z.shape[0]}) are not equal")
        q = z.shape[1]
        zk = None
        if zkeep is not None:
            zk = np.ascontiguousarray(zkeep, dtype=np.uint8)
            if zk.shape[0] != q:
                raise _lib.DimensionMismatch(_lib.IHTB_EDIM, f"zkeep must have length {q} but was {zk.shape[0]}")
        self.comm = comm
        self.p_global = int(p_global) if (comm is not None and p_global is not None) else x.p
        self.x, self.n, self.p, self.q, self.d = x, n, self.p_global, q, d
        if est_r not in EST_R_ID:
            raise ValueError(f"Only support method is Newton or MM, but got {est_r}")
        if est_r != "None" and d != NEGBIN:
            raise _lib.IHTBError(_lib.IHTB_EINVAL, "Only negative binomial regression currently supports nuisance "
                                                   "parameter estimation")
        # a vector k = per-group sparsity `ks`, and then v.k = 0 (src/data_structures.jl:75-81)
        ks = None
        if not np.isscalar(k):
            ks = np.ascontiguousarray(k, dtype=np.int64)
            k = 0
        self.cfg = Cfg(DIST_ID[d], LINK_ID[l], int(k), float(nb_r), float(tol), int(max_iter), int(min_iter),
                       int(max_step), int(sweep_mode), EST_R_ID[est_r], 1 if debias else 0)
        zf = np.asfortranarray(z)
        self._h = C.c_void_p()
        # a SHARD multi-device operator runs the same calls through ihtb_mfit_* (one host thread per device inside)
        self._multi = isinstance(x, B200MultiSnpLinAlg)
        self._pre = "ihtb_mfit_" if self._multi else "ihtb_fit_"
        if self._multi:
            if x.mode != B200MultiSnpLinAlg.SHARD:
                raise _lib.IHTBError(_lib.IHTB_EINVAL, "fit_iht over several GPUs needs a SHARD multi-device operator")
            check(load().ihtb_mfit_create(x._h, ptr(y, C.c_double), zf.ctypes.data_as(C.POINTER(C.c_double)), q,
                                          ptr(zk, C.c_uint8) if zk is not None else None, C.byref(self.cfg),
                                          C.byref(self._h)))
        else:
            check(load().ihtb_fit_create_sharded(x._h, comm._h if comm is not None else None, self.p_global,
                                                 ptr(y, C.c_double), zf.ctypes.data_as(C.POINTER(C.c_double)), q,
                                                 ptr(zk, C.c_uint8) if zk is not None else None, C.byref(self.cfg),
                                                 C.byref(self._h)))
        if group is not None and len(group) > 0:
            grp = np.ascontiguousarray(group, dtype=np.int32)
            try:
                if grp.shape[0] != self.p_global:      # src/data_structures.jl:67-69
                    raise _lib.DimensionMismatch(_lib.IHTB_EDIM,
                                                 f"group must have length {self.p_global} but was {grp.shape[0]}")
                check(self._fn("set_groups")(self._h, grp.ctypes.data_as(C.POINTER(C.c_int32)), int(J),
                                                 ptr(ks, C.c_int64) if ks is not None else None,
                                                 0 if ks is None else ks.shape[0]))
            except Exception:
                self.close()
                raise
        elif ks is not None:
            self.close()
            raise AssertionError("Doubly sparse projection specified (since k is a vector) but there are no group "
                                 "information.")
        if weight is not None and len(weight) > 0:
            w = f64(weight)
            if w.shape[0] != self.p_global:       # src/data_structures.jl:71-73
                self.close()
                raise _lib.DimensionMismatch(_lib.IHTB_EDIM,
                                             f"weight must have length {self.p_global} but was {w.shape[0]}")
            try:
                check(self._fn("set_weights")(self._h, ptr(w, C.c_double)))
            except Exception:
                self.close()
                raise

    def _fn(self, name):
        return getattr(load(), self._pre + name)

    def set_k(self, k):
        check(self._fn("set_k")(self._h, int(k)))
        self.cfg.k = int(k)

    def init_iht_indices(self, train_mask=None, init_beta=False):
        m = None if train_mask is None else np.ascontiguousarray(train_mask, dtype=np.uint8)
        mp = ptr(m, C.c_uint8) if m is not None else None
        if self._multi:
            check(load().ihtb_mfit_init(self._h, mp, 1 if init_beta else 0))
        else:
            check((load().ihtb_fit_init_beta if init_beta else load().ihtb_fit_init)(self._h, mp))

    def timer(self, which: int) -> float:
        """CUDA-event stopwatch on the fit stream(s): which=0 start, 1 stop -> elapsed device ms (slowest device)."""
        ms = C.c_double(0.0)
        check(self._fn("timer")(self._h, int(which), C.byref(ms)))
        return ms.value

    def fit(self, trace_cap=None):
        cap = int(self.cfg.max_iter) if trace_cap is None else trace_cap
        res = Result()
        tr = (IterTrace * max(cap, 1))()
        check(self._fn("run")(self._h, C.byref(res), tr, cap))
        n_it = min(int(res.n_steps), cap)
        trace = [(tr[i].logl, tr[i].backtracks, tr[i].tol, tr[i].eta, tr[i].n_candidates) for i in range(n_it)]
        return res, trace

    def get_sparse(self) -> SparseCoef:
        nnz = C.c_int64(0)
        check(self._fn("get_sparse")(self._h, None, None, 0, C.byref(nnz)))
        idx = np.empty(max(nnz.value, 1), dtype=np.int64); val = np.empty(max(nnz.value, 1))
        check(self._fn("get_sparse")(self._h, ptr(idx, C.c_int64), ptr(val, C.c_double), nnz.value, C.byref(nnz)))
        return SparseCoef(self.p, idx[:nnz.value], val[:nnz.value])

    def get(self, mu=False, xb=False, sparse=False):
        """(beta, c, mu, xb); sparse=True returns beta as a `SparseCoef` (no length-p vector is written)."""
        sp = self.get_sparse()
        beta = sp if sparse else sp.dense()
        c = np.empty(self.q)
        m = np.empty(self.n) if mu else None
        x = np.empty(self.n) if xb else None
        check(self._fn("get")(self._h, None, ptr(c, C.c_double),
                              ptr(m, C.c_double) if mu else None, ptr(x, C.c_double) if xb else None))
        return beta, c, m, x

    def predict(self, test_mask=None) -> float:
        m = None if test_mask is None else np.ascontiguousarray(test_mask, dtype=np.uint8)
        dev = C.c_double(0.0)
        check(self._fn("predict")(self._h, ptr(m, C.c_uint8) if m is not None else None, C.byref(dev)))
        return float(dev.value)

    def close(self):
        if getattr(self, "_h", None):
            self._fn("destroy")(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


@dataclass
class mIHTResult:
    """`mIHTResult` (src/data_structures.jl:263-275)."""
    time: float
    logl: float
    iter: int
    beta: np.ndarray      # r x p
    c: np.ndarray         # r x q
    k: int
    traits: int
    Sigma: np.ndarray
    sigma_g: np.ndarray
    trace: list = field(default_factory=list)
    n_sweeps: int = 0
    n_backtracks: int = 0
    sweep_seconds: float = 0.0
    n_launches: int = 0


def is_multivariate(y) -> bool:
    """`is_multivariate` (src/multivariate.jl:481-483)."""
    y = np.asarray(y)
    return y.ndim == 2 and y.shape[0] > 1 and y.shape[1] > 1


class mIHTVariable:
    """`mIHTVariable` (src/data_structures.jl:140-180).  Reference layout on the Python side: Y is r x n, Z is q x n
    (samples are columns); `x` is the n x p genotype operator whose transpose the reference passes."""

    def __init__(self, x: B200SnpLinAlg, z, y, k, zkeep=None, tol=1e-4, max_iter=200, min_iter=5, max_step=3,
                 sweep_mode=_lib.SWEEP_FAST, comm=None, p_global=None):
        Y = np.asarray(y, dtype=np.float64)
        Z = np.asarray(z, dtype=np.float64)
        if Z.ndim == 1:
            Z = Z.reshape(1, -1)
        r, n = Y.shape
        if not (n == x.n == Z.shape[1]):
            raise _lib.DimensionMismatch(
                _lib.IHTB_EDIM, f"number of samples in y, x, and z = {n}, {x.n}, {Z.shape[1]} are not equal")
        q = Z.shape[0]
        if zkeep is not None:
            zk = np.asarray(zkeep, dtype=bool)
            if zk.shape[0] != q:
                raise _lib.DimensionMismatch(_lib.IHTB_EDIM, f"zkeep must have length {q} but was {zk.shape[0]}")
            if not zk.all():
                raise NotImplementedError("multivariate zkeep with false entries is ill-defined in the reference")
        self.x, self.n, self.p, self.q, self.r = x, n, x.p, q, r
        self.cfg = Cfg(0, 0, int(k), 1.0, float(tol), int(max_iter), int(min_iter), int(max_step), int(sweep_mode),
                       0, 0)
        Yc = np.asfortranarray(Y.T)      # n x r column-major
        Zc = np.asfortranarray(Z.T)      # n x q column-major
        self._h = C.c_void_p()
        # a SHARD multi-device operator runs the same calls through ihtb_mmvfit_* (one host thread per device inside)
        self._multi = isinstance(x, B200MultiSnpLinAlg)
        self._pre = "ihtb_mmvfit_" if self._multi else "ihtb_mvfit_"
        if self._multi and x.mode != B200MultiSnpLinAlg.SHARD:
            raise _lib.IHTBError(_lib.IHTB_EINVAL, "fit_iht over several GPUs needs a SHARD multi-device operator")
        self.p_global = int(p_global) if (comm is not None and p_global is not None) else x.p
        if comm is not None:       # one process per GPU: this rank holds columns [x.j0, x.j0 + x.p) of p_global
            if self._multi:
                raise _lib.IHTBError(_lib.IHTB_EINVAL, "a multi-device operator already shards inside one process")
            check(load().ihtb_mvfit_create_sharded(x._h, comm._h, self.p_global, Yc.ctypes.data_as(C.POINTER(C.c_double)),
                                                   r, Zc.ctypes.data_as(C.POINTER(C.c_double)), q, C.byref(self.cfg),
                                                   C.byref(self._h)))
        else:
            check(self._fn("create")(x._h, Yc.ctypes.data_as(C.POINTER(C.c_double)), r,
                                     Zc.ctypes.data_as(C.POINTER(C.c_double)), q, C.byref(self.cfg), C.byref(self._h)))

    def _fn(self, name):
        return getattr(load(), self._pre + name)

    def set_k(self, k):
        check(self._fn("set_k")(self._h, int(k)))

    def init_iht_indices(self, train_mask=None, init_beta=False):
        m = None if train_mask is None else np.ascontiguousarray(train_mask, dtype=np.uint8)
        mp = ptr(m, C.c_uint8) if m is not None else None
        if self._multi:
            check(load().ihtb_mmvfit_init(self._h, mp, 1 if init_beta else 0))
        else:
            check((load().ihtb_mvfit_init_beta if init_beta else load().ihtb_mvfit_init)(self._h, mp))

    def fit(self, trace_cap=None):
        cap = int(self.cfg.max_iter) if trace_cap is None else trace_cap
        res = Result()
        tr = (IterTrace * max(cap, 1))()
        check(self._fn("run")(self._h, C.byref(res), tr, cap))
        n_it = min(int(res.n_steps), cap)
        return res, [(tr[i].logl, tr[i].backtracks, tr[i].tol, tr[i].eta, tr[i].n_candidates) for i in range(n_it)]

    def get(self):
        beta = np.empty((self.r, self.p_global), order="F"); c = np.empty((self.r, self.q), order="F")
        S = np.empty((self.r, self.r)); sg = np.empty(self.r)
        check(self._fn("get")(self._h, beta.ctypes.data_as(C.POINTER(C.c_double)),
                              c.ctypes.data_as(C.POINTER(C.c_double)), ptr(S, C.c_double), ptr(sg, C.c_double)))
        return np.ascontiguousarray(beta), np.ascontiguousarray(c), S, sg

    def predict(self, test_mask=None) -> float:
        m = None if test_mask is None else np.ascontiguousarray(test_mask, dtype=np.uint8)
        out = C.c_double(0.0)
        check(self._fn("predict")(self._h, ptr(m, C.c_uint8) if m is not None else None, C.byref(out)))
        return float(out.value)

    def close(self):
        if getattr(self, "_h", None):
            self._fn("destroy")(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _fit_mv(y, x, z, k, zkeep, tol, max_iter, min_iter, max_step, sweep_mode, init_beta=False, comm=None,
            p_global=None) -> mIHTResult:
    if z is None:
        z = np.ones((1, x.n))
    v = mIHTVariable(x, z, y, k, zkeep, tol, max_iter, min_iter, max_step, sweep_mode, comm, p_global)
    try:
        v.init_iht_indices(None, init_beta)
        res, trace = v.fit()
        beta, c, S, sg = v.get()
    finally:
        v.close()
    return mIHTResult(res.time, res.logl, int(res.iter), beta, c, k, v.r, S, sg, trace, int(res.n_sweeps),
                      int(res.n_backtracks), res.sweep_seconds, int(res.n_launches))


def _check_args(k, max_iter, max_step, tol):
    # the reference's @assert lines (src/fit.jl:87-90, src/utilities.jl:913)
    if max_iter < 0:
        raise AssertionError("Value of max_iter must be nonnegative!\n")
    if max_step < 0:
        raise AssertionError("Value of max_step must be nonnegative!\n")
    if not tol > np.finfo(np.float64).eps:
        raise AssertionError("Value of global tol must exceed machine precision!\n")
    if np.isscalar(k) and k < 0:
        raise AssertionError("Value of k (max predictors per group) must be nonnegative!\n")


def fit_iht(y, x: B200SnpLinAlg, z=None, k=10, d=NORMAL, l=None, zkeep=None, est_r="None", nb_r=1.0, tol=1e-4,
            max_iter=200, min_iter=5, max_step=3, sweep_mode=_lib.SWEEP_FAST, verbose=False, io=None,
            comm=None, p_global=None, init_beta=False, weight=None, debias=False, use_maf=False, J=1,
            group=None) -> IHTResult:
    """`fit_iht(y, x, z; k, d, l, weight, zkeep, est_r, debias, tol, max_iter, min_iter, max_step, init_beta)`
    (src/fit.jl:60-118).  `use_maf` is accepted and, like in the reference, only reported (src/fit.jl:72,108):
    pass `weight=maf_weights(x)` to weight the projection by allele frequency."""
    _check_args(k, max_iter, max_step, tol)
    if J < 0:
        raise AssertionError("Value of J (max number of groups) must be nonnegative!\n")
    if is_multivariate(y):      # d = MvNormal: Y is r x n, Z is q x n (src/fit.jl:66,125)
        if isinstance(x, B200DenseLinAlg):
            raise _lib.IHTBError(_lib.IHTB_EUNSUPPORTED, "multivariate (MvNormal) fits need a B200SnpLinAlg: dense "
                                                         "matrices serve univariate traits only")
        if debias:
            raise _lib.IHTBError(_lib.IHTB_EUNSUPPORTED,
                                 "Currently the debiasing routine for multivariate IHT is broken, sorry!")
        return _fit_mv(y, x, z, k, zkeep, tol, max_iter, min_iter, max_step, sweep_mode, init_beta, comm, p_global)
    if isinstance(x, B200SnpLinAlg) and not x.center:      # the reference checks SnpLinAlg only (src/fit.jl:97-101)
        raise _lib.IHTBError(_lib.IHTB_EUNSUPPORTED, "x is not centered! Please construct SnpLinAlg{Float64}"
                                                     "(::SnpArray, center=true, scale=true)")
    if z is None:
        z = np.ones(x.n)
    l = l or "IdentityLink"
    v = IHTVariable(x, z, y, k, d, l, zkeep, nb_r, tol, max_iter, min_iter, max_step, sweep_mode, comm, p_global,
                    est_r, weight, debias, J, group)
    try:
        v.init_iht_indices(None, init_beta)
        res, trace = v.fit()
        beta, c, _, _ = v.get(sparse=True)              # IHTResult builds the dense vector on first access
    finally:
        v.close()
    if verbose:
        import sys
        out = io or sys.stdout
        for i, t in enumerate(trace):
            print(f"Iteration {i + 1}: loglikelihood = {t[0]}, backtracks = {t[1]}, tol = {t[2]}", file=out)
    return IHTResult(res.time, res.logl, int(res.iter), beta, c, J, k, [] if group is None else list(group), d,
                     res.sigma_g, trace, int(res.n_sweeps),
                     int(res.n_backtracks), res.sweep_seconds, int(res.n_launches))


def maf_weights(x: B200SnpLinAlg, max_weight: float = np.inf) -> np.ndarray:
    """`maf_weights(x; max_weight)` (src/utilities.jl:692-697): w_j = 1 / (2 sqrt(p_j (1 - p_j))) clamped to
    [1, max_weight], p_j the minor allele frequency."""
    if isinstance(x, B200DenseLinAlg):
        raise TypeError("maf_weights needs genotypes (a B200SnpLinAlg), like the reference's maf_weights(x::SnpArray)")
    p = x.maf()
    with np.errstate(divide="ignore"):
        w = 1.0 / (2.0 * np.sqrt(p * (1.0 - p)))
    return np.clip(w, 1.0, max_weight)


def allocate_fold_and_k(q: int, path):
    """Fold-major (fold, k) list, folds numbered 1..q (src/cross_validation.jl:217-223)."""
    return [(fold, int(k)) for fold in range(1, q + 1) for k in path]


def meanloss(fitloss, q: int, folds):
    """Fold-size weighted sum of the per-fold losses (src/cross_validation.jl:304-320)."""
    folds = np.asarray(folds)
    ninfold = np.array([(folds == f).sum() for f in range(1, q + 1)])
    pathsize = len(fitloss) // q
    loss = np.zeros(pathsize)
    for j in range(q):
        wfold = ninfold[j] / folds.shape[0]
        for i in range(pathsize):
            loss[i] += fitloss[i + j * pathsize] * wfold
    return loss


def cv_run(y, x: B200SnpLinAlg, z, folds, q: int, path, d=NORMAL, l="IdentityLink", zkeep=None, nb_r=1.0, max_iter=100,
           min_iter=5, sweep_mode=_lib.SWEEP_FAST, weight=None, debias=False, est_r="None"):
    """The whole univariate (fold, k) grid in ONE library call (`ihtb_cv_run`); returns (mses, iters), fold-major."""
    y = f64(y)
    z = np.asarray(z, dtype=np.float64)
    zf = np.asfortranarray(z.reshape(x.n, -1))
    nq = zf.shape[1]
    zk = None if zkeep is None else np.ascontiguousarray(zkeep, dtype=np.uint8)
    fl = np.ascontiguousarray(folds, dtype=np.int32)
    pa = np.ascontiguousarray(list(path), dtype=np.int64)
    cfg = Cfg(DIST_ID[d], LINK_ID[l], int(pa.max()), float(nb_r), 1e-4, int(max_iter), int(min_iter), 3,
              int(sweep_mode), EST_R_ID[est_r], 1 if debias else 0)
    mses = np.zeros(q * pa.shape[0]); iters = np.zeros(q * pa.shape[0], dtype=np.int64)
    w = None if weight is None else f64(weight)
    if isinstance(x, B200MultiSnpLinAlg):      # REPLICATE handle: the grid is farmed over the devices from a work queue
        busy = np.zeros(x.ngpu)
        check(load().ihtb_mcv_run(x._h, ptr(y, C.c_double), zf.ctypes.data_as(C.POINTER(C.c_double)), nq,
                                  ptr(zk, C.c_uint8) if zk is not None else None, C.byref(cfg),
                                  fl.ctypes.data_as(C.POINTER(C.c_int32)), q, ptr(pa, C.c_int64), pa.shape[0],
                                  ptr(w, C.c_double) if w is not None else None, ptr(mses, C.c_double),
                                  ptr(iters, C.c_int64), ptr(busy, C.c_double)))
        cv_run.last_busy_seconds = busy
        return mses, iters
    check(load().ihtb_cv_run(x._h, ptr(y, C.c_double), zf.ctypes.data_as(C.POINTER(C.c_double)), nq,
                             ptr(zk, C.c_uint8) if zk is not None else None, C.byref(cfg),
                             fl.ctypes.data_as(C.POINTER(C.c_int32)), q, ptr(pa, C.c_int64), pa.shape[0],
                             ptr(w, C.c_double) if w is not None else None, ptr(mses, C.c_double), ptr(iters, C.c_int64)))
    return mses, iters


def cv_iht(y, x: B200SnpLinAlg, z=None, d=NORMAL, l=None, path=range(1, 21), q=5, folds=None, zkeep=None,
           nb_r=1.0, max_iter=100, min_iter=5, sweep_mode=_lib.SWEEP_FAST, combos=None, return_grid=False,
           init_beta=False, weight=None, debias=False, J=1, group=None, est_r="None"):
    """`cv_iht` (src/cross_validation.jl:60-131).  `folds` in 1..q (drawn with numpy's default_rng if omitted).
    `combos`: optional subset of grid positions to run (used by the multi-GPU farm, parallel.py)."""
    path = [int(k) for k in path]
    if max(path) > x.p:
        raise ValueError("Sparsity level in `path` cannot be larger than total number of variables")
    if folds is None:
        folds = np.random.default_rng().integers(1, q + 1, size=x.n)
    folds = np.asarray(folds)
    mv = is_multivariate(y)
    if z is None:
        z = np.ones((1, x.n)) if mv else np.ones(x.n)
    l = l or "IdentityLink"
    grid = allocate_fold_and_k(q, path)
    todo = range(len(grid)) if combos is None else combos
    mses = np.zeros(len(grid)); iters = np.zeros(len(grid), dtype=np.int64)
    if mv:
        v = mIHTVariable(x, z, y, max(path), zkeep, 1e-4, max_iter, min_iter, 3, sweep_mode)
    else:
        v = IHTVariable(x, z, y, max(path), d, l, zkeep, nb_r, 1e-4, max_iter, min_iter, 3, sweep_mode,
                        weight=weight, debias=debias, J=J, group=group, est_r=est_r)
    try:
        for i in todo:
            fold, k = grid[i]
            test = folds == fold
            v.set_k(k)
            v.init_iht_indices(~test, init_beta)
            res, _ = v.fit(trace_cap=0)
            iters[i] = res.iter
            mses[i] = v.predict(test)
    finally:
        v.close()
    if return_grid:
        return mses, iters
    return meanloss(mses, q, folds)


# ---- file-level wrappers (reference src/wrapper.jl) ----------------------------------------------------------------
class MissingPhenotype(ValueError):
    """The reference's MissingException for binary / count traits (src/wrapper.jl:193-207)."""


def _read_fam_phenotype(path: str, col: int = 6, d: str = NORMAL) -> np.ndarray:
    """`parse_phenotypes(x::SnpData, col, d)` (src/wrapper.jl:170-207): column `col` (1-based) of the .fam file.
    "-9" / "NA" are missing: quantitative traits (Normal) are imputed with the mean of the observed phenotypes;
    binary and count traits cannot be imputed and raise, like the reference."""
    vals, missing = [], []
    with open(path) as f:
        for i, line in enumerate(f):
            tok = line.split()[col - 1]
            if tok in ("-9", "NA"):
                vals.append(0.0); missing.append(i)
            else:
                vals.append(float(tok))
    y = np.asarray(vals)
    if missing:
        if d != NORMAL:
            raise MissingPhenotype("Missing phenotype detected: automatic imputation is only possible for quantitative "
                                   f"traits, but the trait is {d} (sample {missing[0] + 1} of {path})")
        y[missing] = (y.sum()) / (len(vals) - len(missing))
    return y


def _read_fam_phenotypes_mv(path: str, cols) -> np.ndarray:
    """`parse_phenotypes(x::SnpData, col::AbstractVector{Int}, ::MvNormal)` (src/wrapper.jl:136-162): r x n, every
    trait imputed with its own observed mean."""
    return np.vstack([_read_fam_phenotype(path, int(c), NORMAL) for c in cols])


def parse_covariates(filename: str, exclude_std_idx=(), standardize: bool = True) -> np.ndarray:
    """`parse_covariates` (src/wrapper.jl:228-247): comma separated, first column all ones, every other column not in
    `exclude_std_idx` (1-based) standardised to mean 0 / variance 1 with the n-1 standard deviation."""
    z = np.loadtxt(filename, delimiter=",", dtype=np.float64, ndmin=2)
    std_idx = np.ones(z.shape[1], dtype=bool)
    for i in exclude_std_idx:
        std_idx[i - 1] = False
    if np.all(z[:, 0] == 1):
        std_idx[0] = False
    if standardize:
        n = z.shape[0]
        for j in np.flatnonzero(std_idx):
            mu = z[:, j].sum() / n
            s = 1.0 / np.sqrt(((z[:, j] - mu) ** 2).sum() / (n - 1))
            z[:, j] = (z[:, j] - mu) * s
    return z


def _load_plink(filename: str, phenotypes, d: str):
    fam = filename + ".fam"
    n = sum(1 for _ in open(fam))
    x = B200SnpLinAlg.from_bed_file(filename + ".bed", n)
    if isinstance(phenotypes, (int, np.integer)):
        y = _read_fam_phenotype(fam, int(phenotypes), d)
    elif isinstance(phenotypes, (list, tuple, np.ndarray)):          # phenotypes=[6, 7]: multivariate, r x n
        y = _read_fam_phenotypes_mv(fam, phenotypes)
    else:
        # comma-separated text file, one sample per row (src/wrapper.jl:209-217): several columns = several traits,
        # returned r x n like the reference
        y = np.loadtxt(phenotypes, delimiter=",", dtype=np.float64)
        if y.ndim == 2:
            y = np.ascontiguousarray(y.T) if y.shape[1] > 1 else y[:, 0]
    return x, y


def _bgen_input(filename: str):
    """The BGEN file that `filename` names (it ends in .bgen, or it is a prefix with prefix.bgen and no prefix.bed),
    else None: PLINK input keeps precedence."""
    fn = os.fspath(filename)
    if fn.endswith(".bgen"):
        return fn
    if not os.path.exists(fn + ".bed") and os.path.exists(fn + ".bgen"):
        return fn + ".bgen"
    return None


def _load_input(filename: str, phenotypes, d: str):
    """(x, y) of PLINK or BGEN input.  BGEN dosages are standardized like the reference's dense dosages
    (src/wrapper.jl:406-423); a BGEN file has no .fam, so phenotypes is an array or a comma-separated file."""
    path = _bgen_input(filename)
    if path is None:
        return _load_plink(filename, phenotypes, d)
    if isinstance(phenotypes, (bool, int, np.integer)):
        raise ValueError(f"{path}: BGEN input has no .fam file to take phenotype column {phenotypes} from; pass "
                         f"phenotypes as an array or a comma-separated file")
    if isinstance(phenotypes, (list, tuple, np.ndarray)):
        y = np.asarray(phenotypes, dtype=np.float64)
    else:
        y = np.loadtxt(phenotypes, delimiter=",", dtype=np.float64)
        if y.ndim == 2:
            y = np.ascontiguousarray(y.T) if y.shape[1] > 1 else y[:, 0]
    return B200DenseLinAlg.from_bgen(path, standardize=True), y


def iht(filename: str, k: int, d: str = NORMAL, phenotypes=6, covariates: str = "", summaryfile: str = None,
        betafile: str = None, exclude_std_idx=(), **kwargs) -> IHTResult:
    """`iht(filename, k, d; phenotypes, covariates, ...)` (src/wrapper.jl:52-120) for binary PLINK input: reads
    `filename`.bed/.fam, builds the device genotype operator with center/scale/impute, standardises covariates and
    runs `fit_iht` with the canonical link (LogLink for NegativeBinomial).  Optional text outputs like the reference.
    BGEN input: `filename` ending in .bgen (or a prefix with prefix.bgen and no prefix.bed) is read with
    `B200DenseLinAlg.from_bgen(standardize=True)`; `phenotypes` is then an array or a comma-separated file."""
    x, y = _load_input(filename, phenotypes, d)
    z = np.ones(x.n) if covariates == "" else parse_covariates(covariates, exclude_std_idx)
    if is_multivariate(y):          # src/wrapper.jl:80,84-85: z is transposed to q x n, no distribution / link
        z = np.ones((1, x.n)) if covariates == "" else np.ascontiguousarray(np.asarray(z).reshape(x.n, -1).T)
        return fit_iht(y, x, z, k=k, **kwargs)
    result = fit_iht(y, x, z, k=k, d=d, l=canonicallink(d), **kwargs)
    if summaryfile:
        with open(summaryfile, "w") as f:
            nz = np.flatnonzero(result.beta)
            f.write(f"\nIHT estimated {nz.size} nonzero SNP predictors and {np.count_nonzero(result.c)} "
                    f"non-genetic predictors.\n\nCompute time (sec):     {result.time}\n"
                    f"Final loglikelihood:    {result.logl}\nSNP PVE:                {result.sigma_g}\n"
                    f"Iterations:             {result.iter}\n\nSelected genetic predictors:\n")
            for j in nz:
                f.write(f"{j + 1}\t{result.beta[j]}\n")
    if betafile:
        np.savetxt(betafile, result.beta)
    return result


def cross_validate(filename: str, d: str = NORMAL, path=range(1, 21), q: int = 5, phenotypes=6, covariates: str = "",
                   cv_summaryfile: str = None, exclude_std_idx=(), folds=None, **kwargs) -> np.ndarray:
    """`cross_validate(filename, d; path, q, ...)` (src/wrapper.jl:301-349) for binary PLINK or BGEN input (as `iht`)."""
    x, y = _load_input(filename, phenotypes, d)
    z = np.ones(x.n) if covariates == "" else parse_covariates(covariates, exclude_std_idx)
    if is_multivariate(y):
        z = np.ones((1, x.n)) if covariates == "" else np.ascontiguousarray(np.asarray(z).reshape(x.n, -1).T)
        mse = cv_iht(y, x, z, path=path, q=q, folds=folds, **kwargs)
    else:
        mse = cv_iht(y, x, z, d=d, l=canonicallink(d), path=path, q=q, folds=folds, **kwargs)
    if cv_summaryfile:
        with open(cv_summaryfile, "w") as f:
            f.write("k\tmse\n")
            for kk, mm in zip(path, mse):
                f.write(f"{kk}\t{mm}\n")
    return mse
