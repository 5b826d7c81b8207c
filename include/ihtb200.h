/*
 * ihtb200.h — C ABI of libihtb200.so: the B200 (sm_100a) implementation of MendelIHT.jl's
 * iterative-hard-thresholding hot path over 2-bit PLINK genotypes.
 *
 * The reference (OpenMendel/MendelIHT.jl v1.4.11) has no FFI of its own: its extension point is
 * Julia dispatch on the matrix type M of IHTVariable{T,M} (src/data_structures.jl:4-6).  Each entry
 * point below names the reference call it replaces; julia/MendelIHTB200.jl and INTEGRATION.md show the
 * `ccall` binding a maintainer adds.  All functions return 0 on success or a negative IHTB_E* code;
 * ihtb_last_error() returns the message for the calling thread.  Plain pointers and sizes only.
 *
 * Ownership: the caller owns every host array; the library copies inputs to the device during the
 * call and never retains host pointers.  Handles are opaque and freed by the *_destroy functions.
 * Threading: a genotype handle is immutable and may be shared; a fit handle is single-owner.
 * There is no CPU fallback: without a CUDA device every compute entry point fails with IHTB_ECUDA.
 */
#ifndef IHTB200_H
#define IHTB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- status codes (the Julia shim rethrows the reference's exception types) ------------------- */
#define IHTB_OK          0
#define IHTB_EINVAL     -1   /* AssertionError / ArgumentError  (src/fit.jl:87-90, cross_validation.jl:81-85) */
#define IHTB_EDIM       -2   /* DimensionMismatch               (src/data_structures.jl:63-85) */
#define IHTB_EDOMAIN    -3   /* DomainError                     (src/utilities.jl:554) */
#define IHTB_ENUMERIC   -4   /* ErrorException("Loglikelihood function is NaN|Inf, aborting...") (src/fit.jl:259-260) */
#define IHTB_ECUDA      -5   /* CUDA / NCCL failure, or no device (no CPU fallback) */
#define IHTB_ENOMEM     -6
#define IHTB_EUNSUPPORTED -7

/* ---- enums ------------------------------------------------------------------------------------ */
enum { IHTB_NORMAL = 0, IHTB_BERNOULLI = 1, IHTB_POISSON = 2, IHTB_NEGBIN = 3 };
enum { IHTB_LINK_IDENTITY = 0, IHTB_LINK_LOGIT = 1, IHTB_LINK_LOG = 2, IHTB_LINK_PROBIT = 3,
       IHTB_LINK_CLOGLOG = 4, IHTB_LINK_CAUCHIT = 5, IHTB_LINK_SQRT = 6, IHTB_LINK_INVERSE = 7,
       IHTB_LINK_INVSQ = 8 };
/* X'v sweep arithmetic.  FAST = FP32 byte-LUT partial sums + FP64 cross-slab sums; the fit then
 * re-scores every top-k candidate exactly in FP64, so support / iteration counts do not depend on it.
 * EXACT = FP64 accumulation throughout (slower kernel; what ihtb_xt_v uses for parity checks).
 * PAIR  = two right-hand sides per pass over the matrix (half2 lookup tables, FP32 sums per slab, FP64 across slabs):
 *         the skinny multi-trait X'R of MvNormal fits (src/multivariate.jl:85) and two lock-stepped cross-validation
 *         fits read the matrix once for two vectors.  Error bound 2^-8 ||v - mean||_1 sigma_inv_j per entry; fits still
 *         re-score their candidates in FP64.  A single (or odd last) right-hand side takes the FAST path. */
enum { IHTB_SWEEP_FAST = 0, IHTB_SWEEP_EXACT = 1, IHTB_SWEEP_PAIR = 2 };

typedef struct ihtb_geno ihtb_geno;     /* replaces SnpLinAlg{Float64}(s; center, scale, impute) or a dense Matrix{T} */
typedef struct ihtb_fit ihtb_fit;       /* replaces IHTVariable{Float64, SnpLinAlg} (src/data_structures.jl:4-43) */
typedef struct ihtb_mvfit ihtb_mvfit;   /* replaces mIHTVariable (src/data_structures.jl:140-180) */
typedef struct ihtb_comm ihtb_comm;     /* NCCL communicator for SNP-sharded fits (no reference equivalent) */

/* kwargs of fit_iht / fit_iht! (src/fit.jl:60-82, 145-154) */
typedef struct ihtb_cfg {
    int32_t dist;        /* IHTB_NORMAL ...                                   `d`        */
    int32_t link;        /* IHTB_LINK_*                                       `l`        */
    int64_t k;           /* sparsity                                          `k`        */
    double  nb_r;        /* NegativeBinomial r (starting value when est_r != 0)  `d.r`    */
    double  tol;         /* 1e-4                                              `tol`      */
    int32_t max_iter;    /* 200 (100 in cv_iht)                               `max_iter` */
    int32_t min_iter;    /* 5                                                 `min_iter` */
    int32_t max_step;    /* 3                                                 `max_step` */
    int32_t sweep_mode;  /* IHTB_SWEEP_FAST | IHTB_SWEEP_EXACT (| IHTB_SWEEP_PAIR: multivariate fits) */
    int32_t est_r;       /* 0 = :None, 1 = :MM, 2 = :Newton (NegativeBinomial only)   `est_r`    */
    int32_t debias;      /* 1: refit the support by IRLS when it did not change, iterations >= 5 (src/fit.jl:187-188) */
} ihtb_cfg;

/* IHTResult (src/data_structures.jl:245-258); beta/c are written through ihtb_fit_get */
typedef struct ihtb_result {
    double  time;        /* seconds inside the fit loop (src/fit.jl:157,174,200) */
    double  logl;        /* best loglikelihood                                   */
    int64_t iter;        /* iterations                                           */
    double  sigma_g;     /* PVE  (src/pve.jl:31-33)                              */
    int64_t n_sweeps;    /* full X'r sweeps executed (init + one per iteration)  */
    int64_t n_backtracks;
    double  sweep_seconds; /* device time spent inside the sweep kernels (CUDA events) */
    int64_t n_launches;  /* kernels launched by this fit                         */
    int64_t n_steps;     /* IHT steps taken = trace lines written (iter, or iter-1 on a max_iter exit) */
} ihtb_result;

/* one line of the verbose trace "Iteration i: loglikelihood = .., backtracks = .., tol = .." (src/fit.jl:194) */
typedef struct ihtb_iter_trace {
    double  logl;
    double  tol;
    double  eta;
    int32_t backtracks;
    int32_t n_candidates;  /* columns re-scored exactly by the projection of this iteration */
} ihtb_iter_trace;

/* ---- library ---------------------------------------------------------------------------------- */
int32_t ihtb_version(void);
int32_t ihtb_last_error(char* buf, int64_t cap);
int32_t ihtb_device_count(int32_t* count);
int32_t ihtb_set_device(int32_t device);
int32_t ihtb_launch_count(int64_t* count);   /* kernels launched by this library in this process */

/* ---- genotype operator (SnpArrays.jl SnpLinAlg; constructed at src/wrapper.jl:68-69,318-319) ---- */
/* bed_cols: SNP-major packed columns WITHOUT the 3 magic bytes; column j starts at bed_cols + j*col_stride_bytes. */
int32_t ihtb_geno_create(const uint8_t* bed_cols, int64_t n, int64_t p, int64_t col_stride_bytes,
                         int32_t center, int32_t scale, int32_t impute, ihtb_geno** out);
/* Piecewise ingest (SURVEY.md 8f2): per-chromosome .bed files or sources that are not one mappable array.  create_empty
 * allocates the HBM matrix, load_columns streams PLINK columns [j_first, j_first+ncols) through pinned double buffers
 * (any order, each column exactly once), finalize computes mu/sigma_inv and the missing-sample index.  Every other
 * call returns IHTB_EINVAL on a handle that is not finalized.  ihtb_geno_create = the three in one call. */
int32_t ihtb_geno_create_empty(int64_t n, int64_t p, int32_t center, int32_t scale, int32_t impute, ihtb_geno** out);
int32_t ihtb_geno_load_columns(ihtb_geno* g, const uint8_t* bed_cols, int64_t col_stride_bytes, int64_t j_first,
                               int64_t ncols);
int32_t ihtb_geno_finalize(ihtb_geno* g);
/* Synthetic PLINK matrix generated on the device (mirrors simulate_random_snparray, src/simulate_utilities.jl:23-51):
 * maf_j = clip(0.5*U, 0.01, 0.5), genotype = Bern(maf)+Bern(maf), optional missing rate; counter-based hash keyed by
 * (seed, global column, sample).  Columns [j0, j0+p_local) of a p_global-column matrix (j0=0, p_local=p for one GPU). */
int32_t ihtb_geno_create_synthetic(int64_t n, int64_t p_local, int64_t j0, uint64_t seed, double missing_rate,
                                   ihtb_geno** out);
/* host twin of the device generator: fills out[ncols][ceil(n/4)] with the same bytes (multi-threaded, no GPU needed) */
int32_t ihtb_synth_host(int64_t n, int64_t ncols, int64_t j0, uint64_t seed, double missing_rate, uint8_t* out);
int32_t ihtb_geno_dims(const ihtb_geno* g, int64_t* n, int64_t* p);
int32_t ihtb_geno_stats(const ihtb_geno* g, double* mu, double* sigma_inv, int64_t* n_missing);
/* SnpArrays `counts(s, dims=1)`: counts[4*j + c] = samples of column j with code c (0: 00, 1: 01 = missing, 2: 10, 3: 11) */
int32_t ihtb_geno_counts(const ihtb_geno* g, int64_t* counts_4_by_p);
/* SnpArrays `maf(s)` (used by maf_weights, src/utilities.jl:692-697): (n1 + 2 n2) / (2 n_obs), folded to <= 0.5 */
int32_t ihtb_geno_maf(const ihtb_geno* g, double* maf);
/* bit-exact getindex: out[(j-j0)*(i1-i0) + (i-i0)] = x[i, j] for i in [i0,i1), j in [j0,j1)  (src/utilities.jl:102,735) */
int32_t ihtb_geno_decode(const ihtb_geno* g, int64_t i0, int64_t i1, int64_t j0, int64_t j1, double* out_colmajor);
/* packed bytes of columns [j0,j1), ceil(n/4) bytes each (for generator parity and .bed export) */
int32_t ihtb_geno_packed(const ihtb_geno* g, int64_t j0, int64_t j1, uint8_t* out);
/* mul!(out, Transpose(x), V): V is n x m column-major, out is p x m column-major  (src/utilities.jl:133, src/multivariate.jl:85) */
int32_t ihtb_xt_v(const ihtb_geno* g, const double* V, int64_t m, double* out, int32_t sweep_mode);
/* x[:, idx] * coef: idx are 0-based columns, coef is k x m column-major, out is n x m  (src/utilities.jl:95-111,728-743) */
int32_t ihtb_x_support(const ihtb_geno* g, const int64_t* idx, int64_t k, const double* coef, int64_t m, double* out);
/* measurement hook: the sweep timed alone on a device-resident vector with CUDA events on its own stream;
 * ms_kernel = the dominant kernel, ms_total = kernel + epilogue, both averaged over `reps` launches */
int32_t ihtb_sweep_bench(const ihtb_geno* g, int32_t sweep_mode, int32_t warmup, int32_t reps, double* ms_kernel,
                         double* ms_total);
/* Bytes of packed genotypes one FAST / PAIR sweep streams from HBM for this handle: p * ceil(n/640) * 128 when the handle
 * holds the ternary copy (five dosages per byte, built at creation when memory allows; IHTB_TERN=0/1 forces), else
 * p * ceil(n/512) * 128 (the PLINK 2-bit tiles).  The algorithmic figure of SURVEY.md 8d stays p * ceil(n/4). */
int32_t ihtb_geno_sweep_stream_bytes(const ihtb_geno* g, int64_t* bytes, int32_t* ternary);
/* The ternary copy as it lies in HBM (ihtb_geno_sweep_stream_bytes bytes): slab-major tiles of 640 samples; inside a slab
 * the columns are grouped by four, and the 16 bytes at word position w (0..31) of a group hold the 32-bit words of its four
 * columns, component i = column 4 q + (i ^ (w & 3)); a word packs samples 20 w .. 20 w + 19 of the slab, a byte five dosages
 * in base 3 (d0 + 3 d1 + 9 d2 + 27 d3 + 81 d4, missing -> 0).  Fails with IHTB_EINVAL when the handle holds no copy. */
int32_t ihtb_geno_ternary_tiles(const ihtb_geno* g, uint8_t* out, int64_t out_bytes);
/* Diagnostic / bench: exact FP64 column dots X[:, cols]' v (the re-scoring of top-k candidates) for ncols columns through
 * the nibble-table kernel every univariate fit uses: average device time per call, and the largest difference to the
 * per-column decode kernel relative to the largest value. */
int32_t ihtb_gather_bench(const ihtb_geno* g, int64_t ncols, int32_t reps, double* ms_per_call, double* max_rel_diff);
int32_t ihtb_geno_destroy(ihtb_geno* g);

/* ---- dense design matrix (fit_iht(y, x::AbstractMatrix{T}, z), src/fit.jl:62; T = Float64 or Float32) -------------
 * The same ihtb_geno handle, holding an n x p matrix of real entries instead of 2-bit genotypes: imputed dosages from
 * VCF / BGEN (src/wrapper.jl:406-423, 451-485) or any dense predictors.  Every univariate fit / CV / debias entry point
 * takes it.  x: n x p column-major, column j at x + j*ld elements (ld >= n), element type dtype (stored on the device in
 * that type; every kernel promotes entries exactly to FP64 and computes in FP64).
 * standardize = 0: the matrix is used as given; a non-finite entry fails with IHTB_EDOMAIN at finalize.
 * standardize = 1: standardize_genotypes! on the device: NaN = missing, mu_j = mean of the observed entries (fixed-order
 *   sum), sigma_j = sqrt(mu_j (1 - mu_j/2)), missing -> mu_j, x = (g - mu_j) * (1/sigma_j) (1/sigma_j = 1 if sigma_j = 0):
 *   integer dosages give the bits of ihtb_geno_decode of the same genotypes in a PLINK handle.
 * On a DENSE handle ihtb_geno_stats returns the mu / sigma_inv / missing counts applied (0 / 1 / 0 with standardize = 0),
 * ihtb_geno_decode the stored values, ihtb_geno_sweep_stream_bytes n*p*sizeof(T) with ternary = 0 (2*n*p for
 * IHTB_DENSE_FIX16 below); ihtb_geno_packed,
 * counts, maf, ternary_tiles, gather_bench and set_offset return IHTB_EUNSUPPORTED and load_columns IHTB_EINVAL.
 * Not supported on a DENSE handle (IHTB_EUNSUPPORTED): multivariate fits, SNP-sharded fits, multi-device handles. */
enum { IHTB_DENSE_F64 = 0, IHTB_DENSE_F32 = 1, IHTB_DENSE_FIX16 = 2 };
/* dtype IHTB_DENSE_F64 or IHTB_DENSE_F32 (IHTB_DENSE_FIX16 needs a denominator: ihtb_geno_create_dosage16) */
int32_t ihtb_geno_create_dense(const void* x, int32_t dtype, int64_t n, int64_t p, int64_t ld, int32_t standardize,
                               ihtb_geno** out);
/* piecewise form: create_dense_empty, load_dense_columns for columns [j_first, j_first+ncols) (any order, each column
 * once; x + c*ld is column j_first + c, elements of the handle's storage type), then ihtb_geno_finalize */
int32_t ihtb_geno_create_dense_empty(int64_t n, int64_t p, int32_t dtype, int32_t standardize, ihtb_geno** out);
int32_t ihtb_geno_load_dense_columns(ihtb_geno* g, const void* x, int64_t ld, int64_t j_first, int64_t ncols);
/* Dosages on a fixed-point grid (IHTB_DENSE_FIX16): uint16_t codes, code c stands for the value c / denominator,
 * 1 <= denominator <= 65534 (PLINK 2 dosages: 16384; VCF DS printed with d decimals: 10^d; BGEN 8-bit: 255).  Code
 * IHTB_DOSAGE16_MISSING is a missing entry: allowed only with standardize = 1 (where it plays the role of NaN), otherwise
 * IHTB_EDOMAIN at finalize.  Storage is 2 bytes per entry, and the handle computes exactly what a Float64 handle of the
 * decoded values computes: every kernel that reads an entry uses g = c / D (IEEE FP64 division) and, standardized,
 * x = (g - mu_j) * sigma_inv_j with the operations above; mu_j, sigma_inv_j and the missing counts come out bit for bit
 * those of the Float64 handle.  So ihtb_geno_decode, ihtb_geno_stats, the support matvec, the re-scoring and with them
 * the fitted support, iterations, beta, c and logl equal those of ihtb_geno_create_dense(c / D as FP64, standardize).
 * The X'v sweep reads the codes (ihtb_geno_sweep_stream_bytes: 2 n p) and centres / scales in its epilogue; its values
 * differ from the Float64 handle's in the last bits, within the documented selection bound.  Columns load through
 * ihtb_geno_load_dense_columns (uint16_t elements) followed by ihtb_geno_finalize. */
enum { IHTB_DOSAGE16_MISSING = 65535 };
int32_t ihtb_geno_create_dosage16(const uint16_t* codes, int64_t n, int64_t p, int64_t ld, int32_t denominator,
                                  int32_t standardize, ihtb_geno** out);
int32_t ihtb_geno_create_dosage16_empty(int64_t n, int64_t p, int32_t denominator, int32_t standardize,
                                        ihtb_geno** out);
/* BGEN 1.2 dosages (layout 2): columns [j_first, j_first+ncols) of an unfinalized IHTB_DENSE_FIX16 or IHTB_DENSE_F64
 * handle from the INFLATED probability blocks of ncols variants (decompression stays with the caller).  Block c is
 * blocks[offsets[c] .. offsets[c+1]) (offsets has ncols + 1 entries, non-decreasing) and becomes column j_first + c.
 * A block is uint32 N, uint16 K, uint8 Pmin, Pmax, N ploidy bytes (bit 7 = missing), uint8 phased, uint8 B, then 2 N
 * B-bit values packed least-significant bit first.  With D = 2^B - 1 the dosage of the second allele is code / D,
 * code = b + 2 (D - a - b) unphased (a = P(11), b = P(12)) or 2 D - h1 - h2 phased; allele = 1 counts the first allele
 * (2 D - code).  FIX16 handles store the code and need D == the handle's denominator (so B <= 15); F64 handles store
 * code / D (IEEE FP64 division, any B).  A missing sample is stored as IHTB_DOSAGE16_MISSING / NaN, so it needs
 * standardize = 1 at ihtb_geno_finalize, as for the other loaders.  The blocks are staged through two pinned buffers
 * and decoded on the device (one CTA per block).  Errors name the LOWEST failing block and the reason:
 *   IHTB_EDIM         block N != n
 *   IHTB_EUNSUPPORTED K != 2, or ploidy != 2 on a non-missing sample
 *   IHTB_EINVAL       B = 0, B > 32, 2^B - 1 != the FIX16 denominator, phased flag not 0 / 1, a block shorter than its
 *                     header + ceil(2 N B / 8) bytes; an F32 handle, allele not 1 / 2, decreasing offsets
 *   IHTB_EDOMAIN      unphased a + b > D
 * After an error the contents of the columns of this call are unspecified (load them again or destroy the handle). */
int32_t ihtb_geno_load_bgen_columns(ihtb_geno* g, const uint8_t* blocks, const int64_t* offsets, int64_t j_first,
                                    int64_t ncols, int32_t allele);
/* Host staging batch of ihtb_geno_load_bgen_columns in bytes (whole blocks, at least one per batch; default 64 MiB,
 * restored by bytes <= 0).  Process-wide; a tuning and test knob. */
int32_t ihtb_bgen_set_batch_bytes(int64_t bytes);

/* ---- univariate fit (fit_iht / fit_iht! / init_iht_indices!, src/fit.jl:60-207, src/utilities.jl:366-438) ---- */
/* y[n]; z is n x q column-major with the intercept in column 0; zkeep[q] (0/1) or NULL for all kept. */
int32_t ihtb_fit_create(const ihtb_geno* g, const double* y, const double* z, int64_t q, const uint8_t* zkeep,
                        const ihtb_cfg* cfg, ihtb_fit** out);
/* SNP-sharded fit, one process per GPU: this rank's genotype handle holds global columns [j0, j0+p_local) of a
 * p_global-column matrix (j0 as given to ihtb_geno_create_synthetic / ihtb_geno_set_offset).  y, z and every n-vector
 * are replicated; partial X*beta is all-reduced (NCCL) and per-shard top-k candidates are all-gathered, so every rank
 * returns the same global model.  beta in ihtb_fit_get has p_global entries.  comm == NULL: plain single-GPU fit. */
int32_t ihtb_fit_create_sharded(const ihtb_geno* g, ihtb_comm* comm, int64_t p_global, const double* y,
                                const double* z, int64_t q, const uint8_t* zkeep, const ihtb_cfg* cfg, ihtb_fit** out);
/* prior weights on the SNPs (keyword `weight`, src/fit.jl:69; scale b before project_k!, src/utilities.jl:291-354):
 * weight[p_global] > 0 (the whole vector on every rank of a sharded fit), NULL clears.  Call before ihtb_fit_init.
 * Covariates keep weight 1 (the reference indexes weight[p+1..p+q] out of bounds there). */
int32_t ihtb_fit_set_weights(ihtb_fit* f, const double* weight);
/* doubly sparse projection (keywords J, k, group: src/fit.jl:64-68; project_group_sparse!, src/utilities.jl:613-679):
 * group[p] holds 1-based group ids, at most J groups stay active with at most k predictors each; ks = NULL uses
 * cfg.k for every group, otherwise ks[n_groups] is the per-group maximum (the reference's vector-valued k; cfg.k is
 * then ignored, check_group src/utilities.jl:902-915 applies).  group = NULL clears.  Call before ihtb_fit_init.
 * Works with either sweep mode (per-group candidate lists carry the sweep's error bound and are re-scored in FP64).
 * On a sharded fit `group` still has p_global entries (the whole matrix) on every rank. */
int32_t ihtb_fit_set_groups(ihtb_fit* f, const int32_t* group, int32_t J, const int64_t* ks, int64_t n_groups);
int32_t ihtb_fit_set_k(ihtb_fit* f, int64_t k);                       /* v.k = sparsity (src/cross_validation.jl:110) */
int32_t ihtb_fit_init(ihtb_fit* f, const uint8_t* train_mask);         /* init_iht_indices!; NULL = all samples */
/* init_iht_indices!(v, init_beta = true, ...): beta starts from per-SNP univariate regressions (initialize_beta!,
 * src/utilities.jl:776-842; Normal traits only, like the reference) */
int32_t ihtb_fit_init_beta(ihtb_fit* f, const uint8_t* train_mask);
int32_t ihtb_fit_run(ihtb_fit* f, ihtb_result* result, ihtb_iter_trace* trace, int64_t trace_cap);   /* fit_iht! + pve */
/* any pointer may be NULL; beta[p], c[q], mu[n], xb[n] */
int32_t ihtb_fit_get(const ihtb_fit* f, double* beta, double* c, double* mu, double* xb);
/* The same model as (global column, coefficient) pairs in column order: *nnz of them exist, at most cap are written
 * (idx / val may be NULL to ask for the count).  For callers that hold a zero-initialised beta[p] (IHTResult.beta is dense,
 * src/data_structures.jl:245-258): scattering k entries replaces writing p doubles. */
int32_t ihtb_fit_get_sparse(const ihtb_fit* f, int64_t* idx, double* val, int64_t cap, int64_t* nnz);
int32_t ihtb_fit_predict(ihtb_fit* f, const uint8_t* test_mask, double* deviance);   /* predict! (src/cross_validation.jl:279-286) */
/* CUDA-event stopwatch on the fit's stream: which=0 start, which=1 stop (elapsed device milliseconds in *ms) */
int32_t ihtb_fit_timer(ihtb_fit* f, int32_t which, double* ms);
/* measurement hook: host wall-clock seconds in [stepsize, gradstep, update_xb+loglikelihood, score+sweep] */
int32_t ihtb_fit_phase_times(const ihtb_fit* f, double* out4);
int32_t ihtb_fit_destroy(ihtb_fit* f);

/* ---- multivariate Normal fit (mIHTVariable, src/multivariate.jl; fit_iht(Y, Transpose(xla), Z), src/fit.jl:60-118) ----
 * Y is n x r column-major (one trait per column; the reference stores r x n), z is n x q column-major with the
 * intercept first, 2 <= r <= 20, every covariate kept.  cfg->k counts non-zero ENTRIES of the r x p matrix B
 * (src/data_structures.jl:233); cfg->dist / link are ignored.  cfg->sweep_mode = IHTB_SWEEP_PAIR reads the matrix once
 * per two traits (the skinny X'R of src/multivariate.jl:85). */
int32_t ihtb_mvfit_create(const ihtb_geno* g, const double* Y, int64_t r, const double* z, int64_t q,
                          const ihtb_cfg* cfg, ihtb_mvfit** out);
/* SNP-sharded form, like ihtb_fit_create_sharded: this rank's handle holds columns [j0, j0 + p_local) of p_global; B
 * in ihtb_mvfit_get has r x p_global entries. */
int32_t ihtb_mvfit_create_sharded(const ihtb_geno* g, ihtb_comm* comm, int64_t p_global, const double* Y, int64_t r,
                                  const double* z, int64_t q, const ihtb_cfg* cfg, ihtb_mvfit** out);
int32_t ihtb_mvfit_set_k(ihtb_mvfit* f, int64_t k);
int32_t ihtb_mvfit_init(ihtb_mvfit* f, const uint8_t* train_mask);
/* init_beta = true (src/multivariate.jl:425-429, initialize_beta! :519-558): B starts from per-trait univariate regressions */
int32_t ihtb_mvfit_init_beta(ihtb_mvfit* f, const uint8_t* train_mask);
int32_t ihtb_mvfit_run(ihtb_mvfit* f, ihtb_result* result, ihtb_iter_trace* trace, int64_t trace_cap);
/* beta: r x p column-major (trait fastest, like Julia's best_B); c: r x q column-major; Sigma: r x r = inv(Gamma);
 * sigma_g[r]: per-trait PVE (src/pve.jl:35-37).  Any pointer may be NULL. */
int32_t ihtb_mvfit_get(const ihtb_mvfit* f, double* beta, double* c, double* Sigma, double* sigma_g);
int32_t ihtb_mvfit_predict(ihtb_mvfit* f, const uint8_t* test_mask, double* mse);   /* src/cross_validation.jl:288-299 */
int32_t ihtb_mvfit_destroy(ihtb_mvfit* f);

/* cv_iht in one call (src/cross_validation.jl:60-131): folds[n] in 1..nfolds, path[npath] sparsity levels; every
 * (fold, k) fit masks the fold out, then mses[(fold-1)*npath + t] = out-of-fold deviance (predict!, :279-286) and
 * iters (optional) the iteration counts.  cfg.k is ignored, cfg.max_iter is the reference's max_iter = 100 default's
 * slot.  weight may be NULL.  The caller applies meanloss (:304-320). */
int32_t ihtb_cv_run(const ihtb_geno* g, const double* y, const double* z, int64_t q, const uint8_t* zkeep,
                    const ihtb_cfg* cfg, const int32_t* folds, int32_t nfolds, const int64_t* path, int64_t npath,
                    const double* weight, double* mses, int64_t* iters);

/* ---- several GPUs driven by ONE process (SURVEY.md 8b `ngpu`: what a Julia caller of fit_iht / cv_iht binds) ----------
 * A multi-device genotype operator over `ngpu` devices (devices = NULL: ordinals 0..ngpu-1; at most 8):
 *   IHTB_MULTI_SHARD     SNP columns block-partitioned over the devices; ihtb_mfit_* then run ONE fit over all of them
 *                        (BASELINE configs[4]): one host thread per device inside each call, X*beta partials all-reduced
 *                        and top-k candidates all-gathered by peer-memory kernels over NVLink (no NCCL, no torchrun);
 *   IHTB_MULTI_REPLICATE the whole matrix on every device; ihtb_mcv_run farms the (fold, k) grid of cv_iht over them
 *                        (BASELINE configs[2]; the reference's Threads.@threads loop, src/cross_validation.jl:98-121).
 * The devices must be able to map each other's memory (NVLink / PCIe peer access); otherwise IHTB_ECUDA. */
enum { IHTB_MULTI_SHARD = 0, IHTB_MULTI_REPLICATE = 1 };
typedef struct ihtb_mgeno ihtb_mgeno;   /* SnpLinAlg over several GPUs */
typedef struct ihtb_mfit ihtb_mfit;     /* IHTVariable over a SHARD handle */
int32_t ihtb_mgeno_create(const uint8_t* bed_cols, int64_t n, int64_t p, int64_t col_stride_bytes, int32_t center,
                          int32_t scale, int32_t impute, int32_t ngpu, const int32_t* devices, int32_t mode,
                          ihtb_mgeno** out);
int32_t ihtb_mgeno_create_synthetic(int64_t n, int64_t p, uint64_t seed, double missing_rate, int32_t ngpu,
                                    const int32_t* devices, int32_t mode, ihtb_mgeno** out);
int32_t ihtb_mgeno_info(const ihtb_mgeno* g, int32_t* ngpu, int32_t* mode, int64_t* n, int64_t* p);
/* borrowed single-device handle of part i (its device ordinal and, for SHARD, the global index of its first column) */
int32_t ihtb_mgeno_part(const ihtb_mgeno* g, int32_t i, ihtb_geno** part, int32_t* device, int64_t* j0);
int32_t ihtb_mgeno_destroy(ihtb_mgeno* g);
/* the ihtb_fit_* calls over a SHARD handle; arguments as in the single-device calls (weight / group have p entries).
 * result and trace come from device 0 -- every device computes the same global model. */
int32_t ihtb_mfit_create(const ihtb_mgeno* g, const double* y, const double* z, int64_t q, const uint8_t* zkeep,
                         const ihtb_cfg* cfg, ihtb_mfit** out);
int32_t ihtb_mfit_set_weights(ihtb_mfit* f, const double* weight);
int32_t ihtb_mfit_set_groups(ihtb_mfit* f, const int32_t* group, int32_t J, const int64_t* ks, int64_t n_groups);
int32_t ihtb_mfit_set_k(ihtb_mfit* f, int64_t k);
int32_t ihtb_mfit_init(ihtb_mfit* f, const uint8_t* train_mask, int32_t init_beta);
int32_t ihtb_mfit_run(ihtb_mfit* f, ihtb_result* result, ihtb_iter_trace* trace, int64_t trace_cap);
int32_t ihtb_mfit_get(const ihtb_mfit* f, double* beta, double* c, double* mu, double* xb);
int32_t ihtb_mfit_get_sparse(const ihtb_mfit* f, int64_t* idx, double* val, int64_t cap, int64_t* nnz);
int32_t ihtb_mfit_predict(ihtb_mfit* f, const uint8_t* test_mask, double* deviance);
int32_t ihtb_mfit_timer(ihtb_mfit* f, int32_t which, double* ms);     /* slowest device's CUDA-event time */
int32_t ihtb_mfit_destroy(ihtb_mfit* f);
/* the multivariate fit over a SHARD handle (mIHTVariable over several GPUs): same arguments as ihtb_mvfit_* */
typedef struct ihtb_mmvfit ihtb_mmvfit;
int32_t ihtb_mmvfit_create(const ihtb_mgeno* g, const double* Y, int64_t r, const double* z, int64_t q,
                           const ihtb_cfg* cfg, ihtb_mmvfit** out);
int32_t ihtb_mmvfit_set_k(ihtb_mmvfit* f, int64_t k);
int32_t ihtb_mmvfit_init(ihtb_mmvfit* f, const uint8_t* train_mask, int32_t init_beta);
int32_t ihtb_mmvfit_run(ihtb_mmvfit* f, ihtb_result* result, ihtb_iter_trace* trace, int64_t trace_cap);
int32_t ihtb_mmvfit_get(const ihtb_mmvfit* f, double* beta, double* c, double* Sigma, double* sigma_g);
int32_t ihtb_mmvfit_predict(ihtb_mmvfit* f, const uint8_t* test_mask, double* mse);
int32_t ihtb_mmvfit_destroy(ihtb_mmvfit* f);
/* ihtb_cv_run over a REPLICATE handle: fits are taken from a shared queue, largest k first (more iterations);
 * busy_seconds[ngpu] (optional) = wall time each device spent on its share */
int32_t ihtb_mcv_run(const ihtb_mgeno* g, const double* y, const double* z, int64_t q, const uint8_t* zkeep,
                     const ihtb_cfg* cfg, const int32_t* folds, int32_t nfolds, const int64_t* path, int64_t npath,
                     const double* weight, double* mses, int64_t* iters, double* busy_seconds);

/* ---- multi-GPU plumbing, one process per GPU (NCCL over NVLink; rendezvous of the 128-byte id is the host's job, e.g. torch.distributed) ---- */
/* nccl_lib_path may be NULL: $IHTB_NCCL_LIB, then libnccl.so.2 are tried (dlopen at run time, no link-time dependency) */
int32_t ihtb_comm_unique_id(const char* nccl_lib_path, uint8_t* out128);
int32_t ihtb_comm_create(const char* nccl_lib_path, const uint8_t* id128, int32_t rank, int32_t nranks, ihtb_comm** out);
int32_t ihtb_comm_destroy(ihtb_comm* c);
/* counters since creation: collectives served by the library's own peer-memory kernels / NCCL calls (rendezvous only,
 * unless peer mapping is unavailable and NCCL carries the collectives) */
int32_t ihtb_comm_stats(const ihtb_comm* c, int64_t* peer_memory_collectives, int64_t* nccl_calls);
/* collective: average device time (us) of `reps` back-to-back all-reduces of n doubles.  use_p2p = 0: ncclAllReduce,
 * 1: the peer-memory path sharded fits take for this n (push-all up to 262144 elements, two-phase reduce-scatter +
 * all-gather above), 2: force push-all, 3: force two-phase (IHTB_EUNSUPPORTED when peer mapping is unavailable) */
int32_t ihtb_comm_allreduce_bench(ihtb_comm* c, int64_t n, int32_t reps, int32_t use_p2p, double* us_per_op);
int32_t ihtb_geno_set_offset(ihtb_geno* g, int64_t j0);   /* global index of local column 0 for host-uploaded shards */

#ifdef __cplusplus
}
#endif
#endif /* IHTB200_H */
