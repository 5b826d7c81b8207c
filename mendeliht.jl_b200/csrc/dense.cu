// Dense design matrix: an n x p matrix of FP64 or FP32 entries on the device (fit_iht(y, x::AbstractMatrix{T}, z),
// reference src/fit.jl:62; the dense Matrix{Float64} of dosages that the VCF / BGEN wrappers build, src/wrapper.jl:406-485),
// or of 16-bit fixed-point dosage codes (FIX16: code c is the value c / D; see "FIX16 storage" below).
//
// Layout: column-major in the element type given, leading dimension ld = n rounded up to DX_ALIGN rows (1 KB of FP64,
// 512 B of FP32), rows n..ld-1 zero.  Every column starts 16-byte aligned and holds a whole number of 128-bit vectors
// per warp, so the sweep streams it with 128-bit loads and no tail branch.  FP32 entries are promoted exactly to FP64;
// all arithmetic is FP64.  The kernels here are the dense counterparts of the PLINK ones:
//   k_dense_xtv + k_dense_epilogue  X'V (sweep.cu): plain sum_i x_ij v_it -- no centring, the mean of v is not used
//   k_dense_x_support                X[:, idx] * coef (support.cu k_x_support): ascending c, one rounding per add
//   k_dense_gather + _fin            exact column dots of the re-scoring (support.cu xt_gather2)
//   k_dense_moments + _fin           init_beta: sum w x, sum w x^2, sum w y x per column (replaces the class sums)
//   k_dense_decode                   getindex / debias column copy (k_decode, k_decode_cols)
//   k_dense_col_stats                finalize: standardize_genotypes! (src/wrapper.jl:406-423), bound scale
// Every reduction has a fixed order (lane, butterfly, slab / split), no floating-point atomics: results are deterministic.
#include "common.cuh"
#include "topk.cuh"
#include <memory>
#include <mutex>
#include <thread>
#include <unordered_map>
#include <string.h>
#include <type_traits>

namespace ihtb {

constexpr int64_t DX_ALIGN = 128;      // rows: ld is a multiple of this (32 lanes x one 16-byte vector of FP32 = 128 rows)
constexpr int DX_ROWS = 2048;          // rows per sweep slab (a multiple of DX_ALIGN); v of a slab lives in shared memory
constexpr int DX_THREADS = 256;        // 8 warps, one column at a time per warp
constexpr int DX_COLS = 64;            // columns per CTA (8 per warp)
constexpr int DX_UNROLL = 8;           // 16-byte loads in flight per lane (8 warps x 32 lanes x 8 x 16 B = 32 KB per CTA)
constexpr int DG_ROWS = 8192;          // rows per split of the re-scoring / moments kernels (32 per thread)
constexpr int DG_THREADS = 256;

constexpr int64_t FX_ALIGN = 256;      // FIX16 rows: ld is a multiple of this (32 lanes x one 16-byte vector of 8 codes)
constexpr int FX_COLS = 128;           // FIX16 sweep: columns per CTA
constexpr int FX_GROUP = 4;            // FIX16 sweep: columns a warp walks together (one read of v serves 4 FMAs)
constexpr int FX_UNROLL = 2;           // FIX16 sweep: vectors per column in flight per lane (2 x 4 x 16 B)

static inline size_t dense_elem(const ihtb_geno* g) {
    return g->dtype == IHTB_DENSE_F32 ? 4 : g->dtype == IHTB_DENSE_FIX16 ? 2 : 8;
}
static inline bool dense_fix16(const ihtb_geno* g) { return g->dtype == IHTB_DENSE_FIX16; }
static inline int64_t dense_slabs(const ihtb_geno* g) { return ceil_div(g->ld, DX_ROWS); }
static inline int64_t dense_splits(const ihtb_geno* g) { return ceil_div(g->n, DG_ROWS); }

// Error bound of the dense sweep and its re-scoring.  Each output is a sum of products x_ij v_i with one rounding per
// FMA / add; a term passes through at most N roundings of its partial sum, so |computed - exact| <= gamma_N
// sum_i |x_ij v_i| with gamma_N = N u / (1 - N u), u = 2^-53 (Higham, Accuracy and Stability, 2nd ed., eq. 4.4):
//   sweep      N_s = DX_ROWS / 32 sequential FMAs per lane + 5 butterfly adds + n_slabs epilogue adds
//   re-scoring N_r = DG_ROWS / DG_THREADS sequential FMAs + 10 block-tree adds + n_splits finalising adds
// The selection compares a sweep value with re-scored ones, so it needs |sweep - rescored| <= gamma_{N_s} + gamma_{N_r}
// (times the absolute sum); sum_i |x_ij v_i| <= max_i |x_ij| * sum_i |v_i| and sum|v| <= sum|r| + |sum r| (the L1 proxy
// the fit computes), so e_j = coef * dscale_j * (sum|r| + |sum r|) with coef = 2 (N_s + N_r) u: the factor 2 covers
// 1 / (1 - N u) and the FP64 rounding of the bound itself many times over.  At n = 10^5 (49 slabs, 13 splits) this is
// 2 * (69 + 49 + 42 + 13) * 2^-53 = 3.8e-14, at n = 10^6 2.9e-13 -- larger than the PLINK EXACT constant 1e-13.
static double dense_bound_coef(const ihtb_geno* g) {
    const double ns = (double)(DX_ROWS / 32 + 5 + dense_slabs(g));
    const double nr = (double)(DG_ROWS / DG_THREADS + 10 + dense_splits(g));
    return 2.0 * (ns + nr) * 0x1p-53;
}

// Error bound of the FIX16 sweep (k_fix16_xtv + k_dense_epilogue) and its re-scoring.  The re-scoring computes
// sum_i x_i v_i over the doubles every other kernel reads (Fix16Col::load: x_i = g_i = fl(c_i / D), or standardized
// x_i = fl(fl(g_i - mu) * sinv), 0 when missing).  The sweep computes out = fl(sinv * fl(fl(S / D) - fl(mu * fl(V - W))))
// with S = sum_i c_i v_i (missing c_i -> 0), V = sum_i v_i and W = sum over the missing rows of v_i (raw: out = fl(S / D)).
// Write L = sum_i |v_i|, A_j = sinv_j (max_i g_ij + |mu_j|), B_j = max_i |x_ij| and T = sinv (S / D - mu (V - W)), the
// exact value of sum over the observed rows of sinv (c_i / D - mu) v_i.
//  (1) Hot loop: c_i v_i is exact inside the FMA (c_i < 2^16), only the sums round.  A term of S passes through at most
//      N_s = 8 DX_ROWS / 256 lane FMAs + 5 butterfly adds + n_slabs slab adds, so |S~ - S| <= gamma_{N_s} max_i c_i L and,
//      through sinv / D, gamma_{N_s} A L.
//  (2) Epilogue: V~ carries N_v = DX_ROWS / 256 + 10 + n_slabs roundings (per-thread sums, block tree, slabs in order), W~ at
//      most N_m = max_j nmiss_j (in order over the column's missing rows); both are sums of |v_i| <= L, so the mu term is
//      off by sinv |mu| (gamma_{N_v} + gamma_{N_m} + 2u) L <= (...) A L.  The division, the subtraction and the product
//      by sinv round quantities that are each <= A L (1 + O(N u)): 3 u A L.  Cancellation between S / D and mu (V - W)
//      costs nothing more: every error above is relative to these absolute sums, not to the result.
//  (3) The doubles: |x_i - sinv (c_i / D - mu)| <= u sinv g_i + 3 u |x_i| (one rounding of c / D, two of the
//      standardization, second order folded in), so |sum_i x_i v_i - T| <= u A L + 3 u B L; the re-scoring adds
//      gamma_{N_r} B L with N_r as in dense_bound_coef.
// Total: |sweep - rescored| <= (gamma_{N_s} + gamma_{N_v} + gamma_{N_m} + gamma_{N_r} + 9 u) (A + B) L.  dscale_j = A_j + B_j
// (k_dense_col_stats), L <= sum|r| + |sum r| as for the float storage, and coef = 2 (N_s + N_v + N_m + N_r + 9) u: the
// factor 2 covers 1 / (1 - N u), the second-order terms and the rounding of the bound.  A raw handle (mu = 0, sinv = 1,
// x = g, no missing rows) is the special case.  At n = 10^5 with 3 % missing (N_m ~ 3 000) this is 7e-13.
static double fix16_bound_coef(const ihtb_geno* g, int64_t max_nmiss) {
    const double ns = (double)(8 * DX_ROWS / 256 + 5 + dense_slabs(g));
    const double nv = (double)(DX_ROWS / 256 + 10 + dense_slabs(g));
    const double nr = (double)(DG_ROWS / DG_THREADS + 10 + dense_splits(g));
    return 2.0 * (ns + nv + (double)max_nmiss + nr + 9.0) * 0x1p-53;
}

const double* geno_bound_scale(const ihtb_geno* g) { return geno_is_dense(g) ? g->dscale.p : g->sinv.p; }
double geno_bound_coef(const ihtb_geno* g, double plink_coef) { return geno_is_dense(g) ? g->dcoef : plink_coef; }

template <typename T> struct Vec16;
template <> struct Vec16<double> { using V = double2; static constexpr int E = 2; };
template <> struct Vec16<float> { using V = float4; static constexpr int E = 4; };
__device__ __forceinline__ double vget(const double2& v, int e) { return e == 0 ? v.x : v.y; }
__device__ __forceinline__ double vget(const float4& v, int e) {
    return (double)(e == 0 ? v.x : e == 1 ? v.y : e == 2 ? v.z : v.w);
}

// ---- column readers: THE value of entry (i, j), as every kernel but the X'v sweep computes with it -------------------
// raw(j, i): the entry before standardization (NaN = missing); load(j, i): the entry as the model sees it.
// Float storage holds the final (standardized) values: both are the stored entry promoted exactly to FP64.
template <typename T> struct StoredCol {
    T* x;
    int64_t ld;
    __device__ __forceinline__ double raw(int64_t j, int64_t i) const { return (double)x[j * ld + i]; }
    __device__ __forceinline__ double load(int64_t j, int64_t i) const { return raw(j, i); }
};
// FIX16 storage: g = c / D by IEEE division, and standardized exactly as k_dense_col_stats standardizes a float column
// (missing -> mu, (g - mu) * sinv), so a FIX16 handle reads the bits a Float64 handle of the values c / D stores.
struct Fix16Col {
    const uint16_t* x;
    int64_t ld;
    double den;
    const double* mu;
    const double* sinv;
    int standardize;
    __device__ __forceinline__ double raw(int64_t j, int64_t i) const {
        const uint32_t c = x[j * ld + i];
        return c == IHTB_DOSAGE16_MISSING ? __longlong_as_double(0x7ff8000000000000ll) : __ddiv_rn((double)c, den);
    }
    __device__ __forceinline__ double load(int64_t j, int64_t i) const {
        double g = raw(j, i);
        if (!standardize) return g;
        const double m = mu[j];
        if (isnan(g)) g = m;
        return __dmul_rn(__dsub_rn(g, m), sinv[j]);
    }
};

template <typename T> static StoredCol<T> stored_col(const ihtb_geno* g) {
    return StoredCol<T>{reinterpret_cast<T*>(g->dense.p), g->ld};
}
static Fix16Col fix16_col(const ihtb_geno* g) {
    return Fix16Col{reinterpret_cast<const uint16_t*>(g->dense.p), g->ld, (double)g->den, g->mu.p, g->sinv.p,
                    g->standardize};
}
// f(reader) with the handle's reader type
template <typename F> static void with_reader(const ihtb_geno* g, F&& f) {
    if (g->dtype == IHTB_DENSE_F32) f(stored_col<float>(g));
    else if (g->dtype == IHTB_DENSE_FIX16) f(fix16_col(g));
    else f(stored_col<double>(g));
}

// ---- X'V sweep ---------------------------------------------------------------------------------------------------
// grid = (ceil(p / DX_COLS), n_slabs).  The CTA stages rows [r0, r0 + DX_ROWS) of the M right-hand sides in shared memory
// (zero beyond n), then each warp walks its columns: lane l reads 16-byte vectors l, l + 32, ... of the column's slab and
// accumulates x * v with FMAs in that order; a butterfly combines the lanes.  part[(t * n_slabs + slab) * p + j].
template <typename T, int M>
__global__ void __launch_bounds__(DX_THREADS)
k_dense_xtv(const T* __restrict__ x, int64_t ld, int64_t n, int64_t p, const double* __restrict__ v,
            double* __restrict__ part) {
    extern __shared__ double vs[];                         // [M][DX_ROWS]
    using V = typename Vec16<T>::V;
    constexpr int E = Vec16<T>::E;
    const int64_t slab = blockIdx.y, n_slabs = gridDim.y, r0 = slab * DX_ROWS;
    const int rows = (int)(ld - r0 < DX_ROWS ? ld - r0 : DX_ROWS);      // a multiple of DX_ALIGN
    for (int e = threadIdx.x; e < M * DX_ROWS; e += DX_THREADS) {
        const int t = e / DX_ROWS, i = e % DX_ROWS;
        vs[e] = (r0 + i < n) ? v[(int64_t)t * n + r0 + i] : 0.0;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nvec = rows / E;                             // a multiple of 32
    const int64_t jend = min((int64_t)(blockIdx.x + 1) * DX_COLS, p);
    for (int64_t j = (int64_t)blockIdx.x * DX_COLS + warp; j < jend; j += DX_THREADS / 32) {
        const V* xc = reinterpret_cast<const V*>(x + j * ld + r0);
        double acc[M];
#pragma unroll
        for (int t = 0; t < M; ++t) acc[t] = 0.0;
        for (int q0 = lane; q0 < nvec; q0 += 32 * DX_UNROLL) {
            V xv[DX_UNROLL];
#pragma unroll
            for (int u = 0; u < DX_UNROLL; ++u)
                if (q0 + 32 * u < nvec) xv[u] = __ldcs(xc + q0 + 32 * u);      // streamed once: do not keep in L2
#pragma unroll
            for (int u = 0; u < DX_UNROLL; ++u) {
                if (q0 + 32 * u < nvec) {
                    const int i = (q0 + 32 * u) * E;
#pragma unroll
                    for (int e = 0; e < E; ++e) {
                        const double xe = vget(xv[u], e);
#pragma unroll
                        for (int t = 0; t < M; ++t) acc[t] = fma(xe, vs[t * DX_ROWS + i + e], acc[t]);
                    }
                }
            }
        }
#pragma unroll
        for (int t = 0; t < M; ++t) {
            const double a = warp_sum(acc[t]);
            if (lane == 0) part[((int64_t)t * n_slabs + slab) * p + j] = a;
        }
    }
}

// ---- FIX16 X'V sweep: S_j = sum_i c_ij v_i over the codes, centring and scale in the epilogue ----------------------
// grid = (ceil(p / FX_COLS), n_slabs).  As k_dense_xtv, but a warp walks FX_GROUP columns at once over the same rows, so
// each v value read from shared memory feeds FX_GROUP FMAs.  Lane l's 16-byte vector q of a column holds the codes of
// slab rows 256 q + 8 l .. 256 q + 8 l + 7; v is staged permuted so that the lane reads them as four double2 at
// 256 q + 64 h + 2 l (h = 0..3): a warp's double2 reads cover 512 contiguous bytes, no bank conflicts.  A code becomes an
// FP64 exactly with one DADD (2^52 + c - 2^52), the missing code becomes 0 before that.  CTAs of column block 0 also
// write the slab's sum of v (fixed order) to part column p, which the epilogue needs for the centring.
// part[(t * n_slabs + slab) * (p + 1) + j].
__device__ __forceinline__ int fx_vperm(int r) { return (r & ~255) + ((r & 7) >> 1) * 64 + ((r >> 3) & 31) * 2 + (r & 1); }
__device__ __forceinline__ double fx_code(uint32_t c) {
    c = c == IHTB_DOSAGE16_MISSING ? 0u : c;
    return __dsub_rn(__hiloint2double(0x43300000, (int)c), 0x1p52);
}

template <int M>
__global__ void __launch_bounds__(DX_THREADS)
k_fix16_xtv(const uint16_t* __restrict__ x, int64_t ld, int64_t n, int64_t p, const double* __restrict__ v,
            double* __restrict__ part) {
    extern __shared__ __align__(16) double fxv[];          // [M][DX_ROWS], rows permuted by fx_vperm (double2 reads)
    const int64_t slab = blockIdx.y, n_slabs = gridDim.y, r0 = slab * DX_ROWS;
    const int rows = (int)(ld - r0 < DX_ROWS ? ld - r0 : DX_ROWS);      // a multiple of FX_ALIGN
    for (int e = threadIdx.x; e < M * DX_ROWS; e += DX_THREADS) {
        const int t = e / DX_ROWS, r = e % DX_ROWS;
        fxv[t * DX_ROWS + fx_vperm(r)] = (r0 + r < n) ? v[(int64_t)t * n + r0 + r] : 0.0;
    }
    __syncthreads();
    if (blockIdx.x == 0) {                                 // block-uniform
        __shared__ double sh[32];
#pragma unroll
        for (int t = 0; t < M; ++t) {
            double a = 0.0;
            for (int r = threadIdx.x; r < DX_ROWS; r += DX_THREADS) a += fxv[t * DX_ROWS + fx_vperm(r)];
            a = block_sum(a, sh);
            if (threadIdx.x == 0) part[((int64_t)t * n_slabs + slab) * (p + 1) + p] = a;
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nvec = rows / (int)FX_ALIGN;
    const int64_t jend = min((int64_t)(blockIdx.x + 1) * FX_COLS, p);
    for (int64_t j0 = (int64_t)blockIdx.x * FX_COLS + warp * FX_GROUP; j0 < jend; j0 += DX_THREADS / 32 * FX_GROUP) {
        const uint4* xc[FX_GROUP];
#pragma unroll
        for (int c = 0; c < FX_GROUP; ++c)             // columns past p re-read column p - 1 and are not written
            xc[c] = reinterpret_cast<const uint4*>(x + min(j0 + c, p - 1) * ld + r0) + lane;
        double acc[FX_GROUP][M];
#pragma unroll
        for (int c = 0; c < FX_GROUP; ++c)
#pragma unroll
            for (int t = 0; t < M; ++t) acc[c][t] = 0.0;
        for (int q0 = 0; q0 < nvec; q0 += FX_UNROLL) {
            uint4 w[FX_UNROLL][FX_GROUP];
#pragma unroll
            for (int u = 0; u < FX_UNROLL; ++u)
                if (q0 + u < nvec)
#pragma unroll
                    for (int c = 0; c < FX_GROUP; ++c) w[u][c] = __ldcs(xc[c] + 32 * (q0 + u));   // streamed once
#pragma unroll
            for (int u = 0; u < FX_UNROLL; ++u) {
                if (q0 + u < nvec) {
                    const double* vb = fxv + (q0 + u) * 256 + 2 * lane;
#pragma unroll
                    for (int h = 0; h < 4; ++h) {
                        double2 vv[M];
#pragma unroll
                        for (int t = 0; t < M; ++t) vv[t] = *reinterpret_cast<const double2*>(vb + t * DX_ROWS + 64 * h);
#pragma unroll
                        for (int c = 0; c < FX_GROUP; ++c) {
                            const uint32_t wd = h == 0 ? w[u][c].x : h == 1 ? w[u][c].y : h == 2 ? w[u][c].z : w[u][c].w;
                            const double c0 = fx_code(wd & 0xffffu), c1 = fx_code(wd >> 16);
#pragma unroll
                            for (int t = 0; t < M; ++t) {
                                acc[c][t] = fma(c0, vv[t].x, acc[c][t]);
                                acc[c][t] = fma(c1, vv[t].y, acc[c][t]);
                            }
                        }
                    }
                }
            }
        }
#pragma unroll
        for (int c = 0; c < FX_GROUP; ++c)
#pragma unroll
            for (int t = 0; t < M; ++t) {
                const double a = warp_sum(acc[c][t]);
                if (lane == 0 && j0 + c < p) part[((int64_t)t * n_slabs + slab) * (p + 1) + j0 + c] = a;
            }
    }
}

// What the epilogue of a FIX16 sweep adds to the slab sums (den == 0: float storage, nothing).
struct Fix16Epi {
    double den = 0.0;
    int standardize = 0;
    const double* mu = nullptr;
    const double* sinv = nullptr;
    const int64_t* miss_ptr = nullptr;
    const int32_t* miss_idx = nullptr;
    const double* v = nullptr;                             // the right-hand sides, n x m
    int64_t n = 0;
};

// out[t * p + j] = sum of the slab partials in slab order.  FIX16 (fx.den != 0): the partials are sums of codes times v,
// and out = S / D (raw) or sinv (S / D - mu (sum v - sum over the column's missing rows of v)), the slab sums of v in
// part column p.  tf (M = 1, optional): the first stage of the |df| selection exactly as k_sweep_epilogue runs it
// (topk.cuh TopkFuse), with the dense error bound.
__global__ void __launch_bounds__(256)
k_dense_epilogue(const double* __restrict__ part, int64_t n_slabs, int64_t p, int m, double* __restrict__ out,
                 TopkFuse tf, Fix16Epi fx) {
    __shared__ int sh[TOPK_BINS];
    const bool fuse = tf.keyL != nullptr;
    if (fuse) {
        topk_first_kernel_housekeeping(tf.hist_other, tf.st, tf.cand, tf.cand_fill);
        for (int b = threadIdx.x; b < TOPK_BINS; b += blockDim.x) sh[b] = 0;
        __syncthreads();
    }
    const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (j < p) {
        const int64_t ps = fx.den != 0.0 ? p + 1 : p;
        for (int t = 0; t < m; ++t) {
            double a = 0.0;
            for (int64_t s = 0; s < n_slabs; ++s) a += part[((int64_t)t * n_slabs + s) * ps + j];
            if (fx.den != 0.0) {
                a = __ddiv_rn(a, fx.den);
                if (fx.standardize) {
                    double vsum = 0.0, vmiss = 0.0;
                    for (int64_t s = 0; s < n_slabs; ++s) vsum += part[((int64_t)t * n_slabs + s) * ps + p];
                    const double* vt = fx.v + (int64_t)t * fx.n;
                    for (int64_t e = fx.miss_ptr[j]; e < fx.miss_ptr[j + 1]; ++e) vmiss += vt[fx.miss_idx[e]];
                    a = __dmul_rn(fx.sinv[j], __dsub_rn(a, __dmul_rn(fx.mu[j], __dsub_rn(vsum, vmiss))));
                }
            }
            out[(int64_t)t * p + j] = a;
            if (fuse) {
                const double bound = tf.bound_coef * (tf.scal[1] + fabs(tf.scal[0]));
                const double w = tf.wt ? tf.wt[j] : 1.0;
                uint32_t kl, ku;
                topk_make_keys(a, w, tf.scale[j] * bound * w, kl, ku);
                tf.keyL[j] = kl; tf.keyU[j] = ku;
                atomicAdd(&sh[kl >> 21], 1);
            }
        }
    }
    if (fuse) {
        __syncthreads();
        for (int b = threadIdx.x; b < TOPK_BINS; b += blockDim.x)
            if (sh[b]) atomicAdd(&tf.hist[b], sh[b]);
    }
}

template <typename T, int M>
static void launch_dense_xtv(const ihtb_geno* g, const double* dV, double* part, cudaStream_t s) {
    const int smem = M * DX_ROWS * (int)sizeof(double);
    if (smem > 48 * 1024) ensure_dynamic_smem(k_dense_xtv<T, M>, smem);
    dim3 grid((unsigned)ceil_div(g->p, DX_COLS), (unsigned)dense_slabs(g));
    IHTB_LAUNCH((k_dense_xtv<T, M>), grid, DX_THREADS, smem, s, reinterpret_cast<const T*>(g->dense.p), g->ld, g->n,
                g->p, dV, part);
}

template <typename T>
static void dense_partials(const ihtb_geno* g, const double* dV, int m, double* part, cudaStream_t s) {
    switch (m) {
        case 1: launch_dense_xtv<T, 1>(g, dV, part, s); break;
        case 2: launch_dense_xtv<T, 2>(g, dV, part, s); break;
        case 3: launch_dense_xtv<T, 3>(g, dV, part, s); break;
        default: launch_dense_xtv<T, 4>(g, dV, part, s); break;
    }
}

template <int M>
static void launch_fix16_xtv(const ihtb_geno* g, const double* dV, double* part, cudaStream_t s) {
    // the kernel also holds 256 B of static shared memory (the slab sum of v), so M = 3 (exactly 48 KB of v) is over the
    // default limit too: opt in for every M (once per kernel and device)
    const int smem = M * DX_ROWS * (int)sizeof(double);
    ensure_dynamic_smem(k_fix16_xtv<M>, smem);
    dim3 grid((unsigned)ceil_div(g->p, FX_COLS), (unsigned)dense_slabs(g));
    IHTB_LAUNCH((k_fix16_xtv<M>), grid, DX_THREADS, smem, s, reinterpret_cast<const uint16_t*>(g->dense.p), g->ld,
                g->n, g->p, dV, part);
}

// m <= 4 right-hand sides; part: [m][n_slabs][p] (float storage) or [m][n_slabs][p + 1] (FIX16)
static void dense_partials_any(const ihtb_geno* g, const double* dV, int m, double* part, cudaStream_t s) {
    if (dense_fix16(g)) {
        switch (m) {
            case 1: launch_fix16_xtv<1>(g, dV, part, s); break;
            case 2: launch_fix16_xtv<2>(g, dV, part, s); break;
            case 3: launch_fix16_xtv<3>(g, dV, part, s); break;
            default: launch_fix16_xtv<4>(g, dV, part, s); break;
        }
    } else if (g->dtype == IHTB_DENSE_F32) {
        dense_partials<float>(g, dV, m, part, s);
    } else {
        dense_partials<double>(g, dV, m, part, s);
    }
}

static size_t dense_part_size(const ihtb_geno* g, int m) {
    return (size_t)(m * dense_slabs(g) * (g->p + (dense_fix16(g) ? 1 : 0)));
}

// the partial-sum kernel alone (sweep bench): one right-hand side
void dense_sweep_kernel_only(const ihtb_geno* g, const double* dV, DBuf<double>* part, cudaStream_t s) {
    const size_t need = dense_part_size(g, 1);
    if (part->n < need) part->alloc(need);
    dense_partials_any(g, dV, 1, part->p, s);
}

void dense_xt_v(const ihtb_geno* g, const double* dV, int64_t m, double* dOut, cudaStream_t s, DBuf<double>* part,
                const TopkFuse* tf) {
    IHTB_CHECK(!tf || m == 1, IHTB_EINVAL, "fused selection stage: one right-hand side");
    const int64_t n_slabs = dense_slabs(g);
    for (int64_t t0 = 0; t0 < m; t0 += 4) {              // right-hand sides in groups of <= 4 per pass over the matrix
        const int mm = (int)std::min<int64_t>(4, m - t0);
        const size_t need = dense_part_size(g, mm);
        if (part->n < need) part->alloc(need);
        dense_partials_any(g, dV + t0 * g->n, mm, part->p, s);
        Fix16Epi fx;
        if (dense_fix16(g)) {
            fx.den = (double)g->den; fx.standardize = g->standardize; fx.mu = g->mu.p; fx.sinv = g->sinv.p;
            fx.miss_ptr = g->miss_ptr.p; fx.miss_idx = g->miss_idx.p; fx.v = dV + t0 * g->n; fx.n = g->n;
        }
        IHTB_LAUNCH(k_dense_epilogue, (unsigned)ceil_div(g->p, 256), 256, 0, s, part->p, n_slabs, g->p, mm,
                    dOut + t0 * g->p, tf ? *tf : TopkFuse(), fx);
    }
}

// ---- support matvec: out[i, t] = sum_c x[i, idx_c] * coef[c, t], ascending c ------------------------------------
template <typename R, int M>
__global__ void __launch_bounds__(256)
k_dense_x_support(R x, int64_t n, const int64_t* __restrict__ idx, int64_t k, const double* __restrict__ coef,
                  double* __restrict__ out) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    double acc[M];
#pragma unroll
    for (int t = 0; t < M; ++t) acc[t] = 0.0;
    for (int64_t c = 0; c < k; ++c) {
        const double xv = x.load(idx[c], i);
#pragma unroll
        for (int t = 0; t < M; ++t) acc[t] = __dadd_rn(acc[t], __dmul_rn(xv, coef[c + (int64_t)t * k]));
    }
#pragma unroll
    for (int t = 0; t < M; ++t) out[i + (int64_t)t * n] = acc[t];
}

template <typename R>
static void dense_x_support_t(const ihtb_geno* g, R x, const int64_t* d_idx, int64_t k, const double* d_coef, int64_t m,
                              double* d_out, cudaStream_t s) {
    const unsigned grid = (unsigned)ceil_div(g->n, 256);
    for (int64_t t0 = 0; t0 < m;) {
        const int64_t mm = m - t0;
        const double* cf = d_coef + t0 * k;
        double* o = d_out + t0 * g->n;
        if (mm >= 4) { IHTB_LAUNCH((k_dense_x_support<R, 4>), grid, 256, 0, s, x, g->n, d_idx, k, cf, o); t0 += 4; }
        else if (mm == 3) { IHTB_LAUNCH((k_dense_x_support<R, 3>), grid, 256, 0, s, x, g->n, d_idx, k, cf, o); t0 += 3; }
        else if (mm == 2) { IHTB_LAUNCH((k_dense_x_support<R, 2>), grid, 256, 0, s, x, g->n, d_idx, k, cf, o); t0 += 2; }
        else { IHTB_LAUNCH((k_dense_x_support<R, 1>), grid, 256, 0, s, x, g->n, d_idx, k, cf, o); t0 += 1; }
    }
}

void dense_x_support(const ihtb_geno* g, const int64_t* d_idx, int64_t k, const double* d_coef, int64_t m,
                     double* d_out, cudaStream_t s) {
    with_reader(g, [&](auto x) { dense_x_support_t(g, x, d_idx, k, d_coef, m, d_out, s); });
}

// ---- exact column dots (re-scoring): out[c + t * ncols] = sum_i x_ij v_it, j = column c of the two lists ---------
// grid = (ncols, n_splits): the CTA reduces rows [sp * DG_ROWS, ...) of one column (sequential FMAs per thread, fixed
// block tree); k_dense_gather_fin adds the splits in order.  A column index < 0 (unused candidate slot) gives 0.
template <typename R, int M>
__global__ void __launch_bounds__(DG_THREADS)
k_dense_gather(R x, int64_t n, const int64_t* __restrict__ cols, int64_t n_a,
               const int64_t* __restrict__ cols_b, const double* __restrict__ v, double* __restrict__ part) {
    __shared__ double sh[32];
    const int64_t c = blockIdx.x, sp = blockIdx.y;
    const int64_t j = c < n_a ? cols[c] : cols_b[c - n_a];
    if (j < 0) return;                                     // block-uniform
    const int64_t r1 = min((sp + 1) * (int64_t)DG_ROWS, n);
    double a[M];
#pragma unroll
    for (int t = 0; t < M; ++t) a[t] = 0.0;
    for (int64_t i = sp * DG_ROWS + threadIdx.x; i < r1; i += DG_THREADS) {
        const double xv = x.load(j, i);
#pragma unroll
        for (int t = 0; t < M; ++t) a[t] = fma(xv, v[i + (int64_t)t * n], a[t]);
    }
#pragma unroll
    for (int t = 0; t < M; ++t) {
        const double at = block_sum(a[t], sh);
        if (threadIdx.x == 0) part[(c * gridDim.y + sp) * M + t] = at;
    }
}

template <int M>
__global__ void k_dense_gather_fin(const int64_t* __restrict__ cols, int64_t n_a, const int64_t* __restrict__ cols_b,
                                   int64_t ncols, int nsplit, const double* __restrict__ part, double* __restrict__ out) {
    const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (e >= ncols * M) return;
    const int64_t c = e / M;
    const int t = (int)(e % M);
    const int64_t j = c < n_a ? cols[c] : cols_b[c - n_a];
    double a = 0.0;
    if (j >= 0)
        for (int sp = 0; sp < nsplit; ++sp) a = __dadd_rn(a, part[(c * nsplit + sp) * M + t]);
    out[c + (int64_t)t * ncols] = a;
}

// one buffer per stream, as support.cu gather_scratch (fits of several host threads run concurrently)
static DBuf<double>& dense_gather_scratch(cudaStream_t s) {
    static std::mutex mu;
    static std::unordered_map<cudaStream_t, std::unique_ptr<DBuf<double>>> pool;
    std::lock_guard<std::mutex> lk(mu);
    auto& slot = pool[s];
    if (!slot) slot.reset(new DBuf<double>());
    return *slot;
}

template <typename R, int M>
static void launch_dense_gather(const ihtb_geno* g, R x, const int64_t* a, int64_t n_a, const int64_t* b, int64_t ncols,
                                const double* v, double* out, cudaStream_t s) {
    DBuf<double>& sc = dense_gather_scratch(s);
    const int nsplit = (int)dense_splits(g);
    const size_t need = (size_t)ncols * nsplit * M;
    if (sc.n < need) {
        IHTB_CUDA(cudaStreamSynchronize(s));
        sc.alloc(need < 65536 ? 65536 : need);
    }
    IHTB_LAUNCH((k_dense_gather<R, M>), dim3((unsigned)ncols, (unsigned)nsplit), DG_THREADS, 0, s, x, g->n, a, n_a, b,
                v, sc.p);
    IHTB_LAUNCH((k_dense_gather_fin<M>), (unsigned)ceil_div(ncols * M, 128), 128, 0, s, a, n_a, b, ncols, nsplit, sc.p,
                out);
}

template <typename R>
static void dense_gather_t(const ihtb_geno* g, R x, const int64_t* a, int64_t n_a, const int64_t* b, int64_t ncols,
                           const double* d_v, int64_t m, double* d_out, cudaStream_t s) {
    for (int64_t t0 = 0; t0 < m;) {
        const int64_t mm = m - t0;
        const double* vv = d_v + t0 * g->n;
        double* o = d_out + t0 * ncols;
        if (mm >= 4) { launch_dense_gather<R, 4>(g, x, a, n_a, b, ncols, vv, o, s); t0 += 4; }
        else if (mm == 3) { launch_dense_gather<R, 3>(g, x, a, n_a, b, ncols, vv, o, s); t0 += 3; }
        else if (mm == 2) { launch_dense_gather<R, 2>(g, x, a, n_a, b, ncols, vv, o, s); t0 += 2; }
        else { launch_dense_gather<R, 1>(g, x, a, n_a, b, ncols, vv, o, s); t0 += 1; }
    }
}

void dense_xt_gather2(const ihtb_geno* g, const int64_t* d_cols_a, int64_t n_a, const int64_t* d_cols_b, int64_t n_b,
                      const double* d_v, int64_t m, double* d_out, cudaStream_t s) {
    const int64_t ncols = n_a + n_b;
    if (ncols == 0) return;
    with_reader(g, [&](auto x) { dense_gather_t(g, x, d_cols_a, n_a, d_cols_b, ncols, d_v, m, d_out, s); });
}

// ---- init_beta moments: part[(c * nsplit + sp) * 3 + {0,1,2}] = sums of w x, w x^2, wy x over one split -------------
template <typename R>
__global__ void __launch_bounds__(DG_THREADS)
k_dense_moments(R x, int64_t n, const double* __restrict__ w,
                const double* __restrict__ wy, double* __restrict__ part) {
    __shared__ double sh[32];
    const int64_t j = blockIdx.x, sp = blockIdx.y;
    const int64_t r1 = min((sp + 1) * (int64_t)DG_ROWS, n);
    double a = 0.0, b = 0.0, c = 0.0;
    for (int64_t i = sp * DG_ROWS + threadIdx.x; i < r1; i += DG_THREADS) {
        const double xv = x.load(j, i), wi = w[i];
        a = fma(wi, xv, a);
        b = fma(wi, __dmul_rn(xv, xv), b);
        c = fma(wy[i], xv, c);
    }
    a = block_sum(a, sh);
    b = block_sum(b, sh);
    c = block_sum(c, sh);
    if (threadIdx.x == 0) {
        double* o = part + (j * gridDim.y + sp) * 3;
        o[0] = a; o[1] = b; o[2] = c;
    }
}

__global__ void k_dense_moments_fin(int64_t p, int nsplit, const double* __restrict__ part, double* __restrict__ sx,
                                    double* __restrict__ sxx, double* __restrict__ sxy) {
    const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (j >= p) return;
    double a = 0.0, b = 0.0, c = 0.0;
    for (int sp = 0; sp < nsplit; ++sp) {
        const double* o = part + (j * nsplit + sp) * 3;
        a += o[0]; b += o[1]; c += o[2];
    }
    sx[j] = a; sxx[j] = b; sxy[j] = c;
}

void dense_init_beta_moments(const ihtb_geno* g, const double* d_w, const double* d_wy, double* d_sx, double* d_sxx,
                             double* d_sxy, cudaStream_t s) {
    const int nsplit = (int)dense_splits(g);
    DBuf<double> part((size_t)(g->p * nsplit * 3));
    dim3 grid((unsigned)g->p, (unsigned)nsplit);
    with_reader(g, [&](auto x) {
        IHTB_LAUNCH(k_dense_moments<decltype(x)>, grid, DG_THREADS, 0, s, x, g->n, d_w, d_wy, part.p);
    });
    IHTB_LAUNCH(k_dense_moments_fin, (unsigned)ceil_div(g->p, 256), 256, 0, s, g->p, nsplit, part.p, d_sx, d_sxx, d_sxy);
    IHTB_CUDA(cudaStreamSynchronize(s));               // `part` is freed on return
}

// ---- decode: out[c * ni + (i - i0)] = x[i, j_c] in FP64; j_c = cols[c] (cols != NULL; < 0 gives zeros) or j0 + c ----
template <typename R>
__global__ void k_dense_decode(R x, const int64_t* __restrict__ cols, int64_t j0,
                               int64_t ncols, int64_t i0, int64_t ni, double* __restrict__ out) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= ni * ncols) return;
    const int64_t c = t / ni, i = i0 + t % ni;
    const int64_t j = cols ? cols[c] : j0 + c;
    out[t] = j < 0 ? 0.0 : x.load(j, i);
}

static void dense_decode(const ihtb_geno* g, const int64_t* d_cols, int64_t j0, int64_t ncols, int64_t i0, int64_t ni,
                         double* d_out, cudaStream_t s) {
    const int64_t total = ni * ncols;
    if (total == 0) return;
    with_reader(g, [&](auto x) {
        IHTB_LAUNCH(k_dense_decode<decltype(x)>, (unsigned)ceil_div(total, 256), 256, 0, s, x, d_cols, j0, ncols, i0,
                    ni, d_out);
    });
}

void dense_decode_cols(const ihtb_geno* g, const int64_t* d_cols, int64_t k, double* d_out, cudaStream_t s) {
    dense_decode(g, d_cols, 0, k, 0, g->n, d_out, s);
}

// ---- finalize: one CTA per column ---------------------------------------------------------------------------------
// standardize = 1 (standardize_genotypes!, src/wrapper.jl:406-423): NaN = missing, mu = (fixed-order FP64 sum of the
// observed entries) / n_observed, sigma_inv with k_col_stats' operations, x <- ((missing ? mu : x) - mu) * sigma_inv with
// k_decode's operations (so integer dosages reproduce a PLINK handle's decode bit for bit), rounded to T on store.
// standardize = 0: counts the non-finite entries (bad[0]), mu = 0, sigma_inv = 1.  Both: dscale = max_i |x_ij| stored.
// FIX16 (R = Fix16Col): the same statistics from g = c / D (the missing code reads as NaN), nothing is written back, and
// dscale = sinv (max_i g_ij + |mu|) + max_i |x_ij| (fix16_bound_coef).
__device__ __forceinline__ double block_max(double v, double* sh) {    // order-independent: a plain tree
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0)
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) v = fmax(v, sh[w]);
    return v;
}

template <typename R>
__global__ void __launch_bounds__(256)
k_dense_col_stats(R x, int64_t n, int standardize, double* __restrict__ mu, double* __restrict__ sinv,
                  int32_t* __restrict__ nmiss, double* __restrict__ dscale, unsigned long long* __restrict__ bad) {
    constexpr bool stored = !std::is_same<R, Fix16Col>::value;
    __shared__ double sh[32];
    __shared__ double s_m, s_si;
    const int64_t j = blockIdx.x;
    double sum = 0.0, cnt = 0.0, nb = 0.0;      // counts are exact in FP64
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
        const double g = x.raw(j, i);
        if (standardize && !isnan(g)) { sum += g; cnt += 1.0; }
        if (standardize ? isinf(g) : !isfinite(g)) nb += 1.0;
    }
    sum = block_sum(sum, sh);
    cnt = block_sum(cnt, sh);
    nb = block_sum(nb, sh);
    if (threadIdx.x == 0) {
        if (standardize) {
            const double m = sum / cnt;
            const double s = sqrt(__dmul_rn(m, __dsub_rn(1.0, m / 2.0)));
            s_m = m;
            s_si = s > 0.0 ? 1.0 / s : 1.0;
            mu[j] = m; sinv[j] = s_si; nmiss[j] = (int32_t)(n - (int64_t)cnt);
        } else {
            s_m = 0.0; s_si = 1.0;
            mu[j] = 0.0; sinv[j] = 1.0; nmiss[j] = 0;
        }
        if (nb > 0.0) atomicAdd(bad, (unsigned long long)nb);
    }
    __syncthreads();
    const double m = s_m, si = s_si;
    double mx = 0.0, gmx = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
        double g = x.raw(j, i);
        if (!stored && !isnan(g)) gmx = fmax(gmx, g);
        if (standardize) {
            if (isnan(g)) g = m;
            if constexpr (stored) {
                using T = typename std::remove_pointer<decltype(x.x)>::type;
                const T st = (T)__dmul_rn(__dsub_rn(g, m), si);
                x.x[j * x.ld + i] = st;
                g = (double)st;
            } else {
                g = __dmul_rn(__dsub_rn(g, m), si);
            }
        }
        mx = fmax(mx, fabs(g));
    }
    mx = block_max(mx, sh);
    if (!stored) gmx = block_max(gmx, sh);
    if (threadIdx.x == 0) dscale[j] = stored ? mx : si * (gmx + fabs(m)) + mx;
}

// CSR of the missing rows of a standardized FIX16 handle (the centring of k_dense_epilogue): one warp per column, rows
// ascending (ballot compaction), idx[ptr[j] ..] = rows of column j holding IHTB_DOSAGE16_MISSING
__global__ void k_fix16_missing(const uint16_t* __restrict__ x, int64_t ld, int64_t n, int64_t p,
                                const int64_t* __restrict__ ptr, int32_t* __restrict__ idx) {
    const int64_t j = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (j >= p) return;                                    // warp-uniform
    int64_t pos = ptr[j];
    for (int64_t i0 = 0; i0 < n; i0 += 32) {
        const int64_t i = i0 + lane;
        const bool miss = i < n && x[j * ld + i] == IHTB_DOSAGE16_MISSING;
        const unsigned b = __ballot_sync(0xffffffffu, miss);
        if (miss) idx[pos + __popc(b & ((1u << lane) - 1u))] = (int32_t)i;
        pos += __popc(b);
    }
}

static void fix16_missing_rows(ihtb_geno* g, int64_t* max_nmiss) {
    std::vector<int32_t> nm((size_t)g->p);
    IHTB_CUDA(cudaMemcpy(nm.data(), g->nmiss.p, g->p * sizeof(int32_t), cudaMemcpyDeviceToHost));
    std::vector<int64_t> ptr((size_t)g->p + 1, 0);
    *max_nmiss = 0;
    for (int64_t j = 0; j < g->p; ++j) {
        ptr[j + 1] = ptr[j] + nm[j];
        *max_nmiss = std::max<int64_t>(*max_nmiss, nm[j]);
    }
    g->total_missing = ptr[g->p];
    g->miss_ptr.alloc(g->p + 1);
    IHTB_CUDA(cudaMemcpy(g->miss_ptr.p, ptr.data(), (g->p + 1) * sizeof(int64_t), cudaMemcpyHostToDevice));
    if (g->total_missing) {
        g->miss_idx.alloc(g->total_missing);
        IHTB_LAUNCH(k_fix16_missing, (unsigned)ceil_div(g->p * 32, 256), 256, 0, 0,
                    reinterpret_cast<const uint16_t*>(g->dense.p), g->ld, g->n, g->p, g->miss_ptr.p, g->miss_idx.p);
        IHTB_CUDA(cudaStreamSynchronize(0));           // fits read the list from their own streams
    }
}

void dense_finalize(ihtb_geno* g) {
    g->bgen_stage.reset();
    g->mu.alloc(g->p); g->sinv.alloc(g->p); g->nmiss.alloc(g->p); g->dscale.alloc(g->p);
    DBuf<unsigned long long> bad(1);
    bad.zero(0);
    with_reader(g, [&](auto x) {
        IHTB_LAUNCH(k_dense_col_stats<decltype(x)>, (unsigned)g->p, 256, 0, 0, x, g->n, g->standardize, g->mu.p,
                    g->sinv.p, g->nmiss.p, g->dscale.p, bad.p);
    });
    unsigned long long nbad = 0;
    IHTB_CUDA(cudaMemcpy(&nbad, bad.p, sizeof(nbad), cudaMemcpyDeviceToHost));
    if (dense_fix16(g)) {
        IHTB_CHECK(nbad == 0, IHTB_EDOMAIN,
                   std::to_string(nbad) + " entries hold the missing code 65535, which needs standardize = 1");
        int64_t max_nmiss = 0;
        if (g->standardize) fix16_missing_rows(g, &max_nmiss);
        g->dcoef = fix16_bound_coef(g, max_nmiss);
        return;
    }
    IHTB_CHECK(nbad == 0, IHTB_EDOMAIN,
               std::to_string(nbad) + " entries of the dense matrix are not finite (standardize = 1 reads NaN as missing)");
    g->dcoef = dense_bound_coef(g);
}

// Host -> HBM ingest of `ncols` columns (x + c * ld_host is column j_dst + c): two pinned buffers, the host threads
// gather chunk i + 1 while chunk i is copied with one 2-D copy into the padded device columns (like geno.cu
// upload_columns, without a repack: the device layout is the host's with a larger leading dimension).
void dense_upload(ihtb_geno* g, const void* x, int64_t ld_host, int64_t j_dst, int64_t ncols) {
    const size_t es = dense_elem(g), colb = (size_t)g->n * es;
    int64_t cols_per = (int64_t)((size_t(64) << 20) / colb);
    if (cols_per < 1) cols_per = 1;
    if (cols_per > ncols) cols_per = ncols;
    const int NB = 2;
    HBuf<uint8_t> hbuf[NB];
    cudaEvent_t done[NB] = {nullptr, nullptr};
    cudaStream_t st;
    IHTB_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    unsigned nt = std::thread::hardware_concurrency();
    if (nt == 0) nt = 1;
    if (nt > 16) nt = 16;
    const uint8_t* src0 = reinterpret_cast<const uint8_t*>(x);
    int b = 0;
    try {
        for (int i = 0; i < NB; ++i) {
            hbuf[i].alloc((size_t)cols_per * colb);
            IHTB_CUDA(cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming));
        }
        for (int64_t j = 0; j < ncols; j += cols_per, b ^= 1) {
            const int64_t h = std::min<int64_t>(ncols - j, cols_per);
            IHTB_CUDA(cudaEventSynchronize(done[b]));
            uint8_t* dst = hbuf[b].p;
            const uint8_t* src = src0 + (size_t)j * (size_t)ld_host * es;
            const unsigned use = (unsigned)std::min<int64_t>(nt, h);
            auto copy = [=](int64_t c0, int64_t c1) {
                for (int64_t c = c0; c < c1; ++c) memcpy(dst + c * colb, src + (size_t)c * (size_t)ld_host * es, colb);
            };
            std::vector<std::thread> pool;
            for (unsigned t = 1; t < use; ++t) pool.emplace_back(copy, h * t / use, h * (t + 1) / use);
            copy(0, h / use);
            for (auto& th : pool) th.join();
            IHTB_CUDA(cudaMemcpy2DAsync(g->dense.p + (size_t)(j_dst + j) * (size_t)g->ld * es, (size_t)g->ld * es, dst,
                                        colb, colb, (size_t)h, cudaMemcpyHostToDevice, st));
            IHTB_CUDA(cudaEventRecord(done[b], st));
        }
        IHTB_CUDA(cudaStreamSynchronize(st));
    } catch (...) {
        cudaStreamSynchronize(st);
        for (int i = 0; i < NB; ++i) if (done[i]) cudaEventDestroy(done[i]);
        cudaStreamDestroy(st);
        throw;
    }
    for (int i = 0; i < NB; ++i) cudaEventDestroy(done[i]);
    cudaStreamDestroy(st);
}

// den = 0: float storage (dtype F64 / F32); den in [1, 65534]: FIX16 codes with that denominator
ihtb_geno* dense_new_handle(int64_t n, int64_t p, int dtype, int standardize, int32_t den) {
    IHTB_CHECK(n > 0 && p > 0, IHTB_EDIM, "dense matrix must have n > 0 and p > 0");
    IHTB_CHECK(n < (int64_t(1) << 31), IHTB_EDIM, "n must be < 2^31");
    if (den == 0)
        IHTB_CHECK(dtype == IHTB_DENSE_F64 || dtype == IHTB_DENSE_F32, IHTB_EINVAL,
                   "dtype must be IHTB_DENSE_F64 or IHTB_DENSE_F32 (fixed-point dosages: ihtb_geno_create_dosage16)");
    else
        IHTB_CHECK(dtype == IHTB_DENSE_FIX16 && den >= 1 && den <= 65534, IHTB_EINVAL,
                   "the dosage denominator must be in [1, 65534]");
    IHTB_CHECK(standardize == 0 || standardize == 1, IHTB_EINVAL, "standardize must be 0 or 1");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        throw Error(IHTB_ECUDA, "no CUDA device available (libihtb200 has no CPU fallback)");
    std::unique_ptr<ihtb_geno> g(new ihtb_geno());
    g->kind = GENO_DENSE;
    IHTB_CUDA(cudaGetDevice(&g->device));
    IHTB_CUDA(cudaDeviceGetAttribute(&g->sm_count, cudaDevAttrMultiProcessorCount, g->device));
    g->n = n; g->p = p; g->dtype = dtype; g->standardize = standardize; g->den = den;
    const int64_t align = den ? FX_ALIGN : DX_ALIGN;
    g->ld = ceil_div(n, align) * align;
    g->impute = standardize;
    const size_t bytes = (size_t)p * (size_t)g->ld * dense_elem(g.get());
    g->dense.alloc(bytes);
    IHTB_CUDA(cudaMemset(g->dense.p, 0, bytes));               // rows n..ld-1 stay zero
    return g.release();
}

int64_t dense_stream_bytes(const ihtb_geno* g) { return g->n * g->p * (int64_t)dense_elem(g); }

void dense_decode_block(const ihtb_geno* g, int64_t i0, int64_t i1, int64_t j0, int64_t j1, double* d_out) {
    dense_decode(g, nullptr, j0, j1 - j0, i0, i1 - i0, d_out, 0);
}

}  // namespace ihtb

using namespace ihtb;

extern "C" {

int32_t ihtb_geno_create_dense_empty(int64_t n, int64_t p, int32_t dtype, int32_t standardize, ihtb_geno** out) {
    return guard([&] {
        IHTB_CHECK(out, IHTB_EINVAL, "NULL argument");
        ihtb_geno* g = dense_new_handle(n, p, dtype, standardize);
        g->ready = false;
        *out = g;
    });
}

int32_t ihtb_geno_load_dense_columns(ihtb_geno* g, const void* x, int64_t ld, int64_t j_first, int64_t ncols) {
    return guard([&] {
        IHTB_CHECK(g && x, IHTB_EINVAL, "NULL argument");
        IHTB_CHECK(geno_is_dense(g), IHTB_EINVAL, "not a dense handle (PLINK handles take ihtb_geno_load_columns)");
        IHTB_CHECK(!g->ready, IHTB_EINVAL, "handle is already finalized");
        IHTB_CHECK(ld >= g->n, IHTB_EDIM, "ld is smaller than n");
        IHTB_CHECK(j_first >= 0 && ncols >= 0 && j_first + ncols <= g->p, IHTB_EDIM, "column range outside the matrix");
        IHTB_CUDA(cudaSetDevice(g->device));
        if (ncols > 0) dense_upload(g, x, ld, j_first, ncols);
    });
}

int32_t ihtb_geno_create_dense(const void* x, int32_t dtype, int64_t n, int64_t p, int64_t ld, int32_t standardize,
                               ihtb_geno** out) {
    return guard([&] {
        IHTB_CHECK(x && out, IHTB_EINVAL, "NULL argument");
        IHTB_CHECK(ld >= n, IHTB_EDIM, "ld is smaller than n");
        std::unique_ptr<ihtb_geno> g(dense_new_handle(n, p, dtype, standardize));
        dense_upload(g.get(), x, ld, 0, p);
        dense_finalize(g.get());
        g->ready = true;
        *out = g.release();
    });
}

int32_t ihtb_geno_create_dosage16_empty(int64_t n, int64_t p, int32_t denominator, int32_t standardize,
                                        ihtb_geno** out) {
    return guard([&] {
        IHTB_CHECK(out, IHTB_EINVAL, "NULL argument");
        IHTB_CHECK(denominator >= 1 && denominator <= 65534, IHTB_EINVAL, "the dosage denominator must be in [1, 65534]");
        ihtb_geno* g = dense_new_handle(n, p, IHTB_DENSE_FIX16, standardize, denominator);
        g->ready = false;
        *out = g;
    });
}

int32_t ihtb_geno_create_dosage16(const uint16_t* codes, int64_t n, int64_t p, int64_t ld, int32_t denominator,
                                  int32_t standardize, ihtb_geno** out) {
    return guard([&] {
        IHTB_CHECK(codes && out, IHTB_EINVAL, "NULL argument");
        IHTB_CHECK(ld >= n, IHTB_EDIM, "ld is smaller than n");
        IHTB_CHECK(denominator >= 1 && denominator <= 65534, IHTB_EINVAL, "the dosage denominator must be in [1, 65534]");
        std::unique_ptr<ihtb_geno> g(dense_new_handle(n, p, IHTB_DENSE_FIX16, standardize, denominator));
        dense_upload(g.get(), codes, ld, 0, p);
        dense_finalize(g.get());
        g->ready = true;
        *out = g.release();
    });
}

}  // extern "C"
