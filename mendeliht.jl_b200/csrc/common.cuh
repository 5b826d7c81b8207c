// Shared internals of libihtb200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <memory>
#include <string>
#include <vector>
#include <stdexcept>
#include "../../include/ihtb200.h"

namespace ihtb {

// ---- error plumbing: C++ exceptions inside, status codes at the C boundary -------------------
struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};
void set_last_error(const std::string& m);
const std::string& last_error();
struct LaunchCounter {        // relaxed atomic: fits on several host threads (multi-device handles) share it
    int64_t v = 0;
    LaunchCounter& operator++(int) { __atomic_fetch_add(&v, 1, __ATOMIC_RELAXED); return *this; }
    operator int64_t() const { return __atomic_load_n(&v, __ATOMIC_RELAXED); }
};
LaunchCounter& launch_counter();
bool debug_sync();   // IHTB_DEBUG_SYNC=1: synchronise and check after every kernel launch

#define IHTB_CUDA(call)                                                                      \
    do {                                                                                     \
        cudaError_t e__ = (call);                                                            \
        if (e__ != cudaSuccess)                                                              \
            throw ::ihtb::Error(IHTB_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e__)); \
    } while (0)

#define IHTB_CHECK(cond, code, msg)                                  \
    do {                                                             \
        if (!(cond)) throw ::ihtb::Error((code), (msg));             \
    } while (0)

// every kernel launch goes through this so `gpu_launches` in bench.py is a real count
#define IHTB_LAUNCH(kernel, grid, block, smem, stream, ...)          \
    do {                                                             \
        kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__);  \
        ::ihtb::launch_counter()++;                                  \
        IHTB_CUDA(cudaGetLastError());                               \
        if (::ihtb::debug_sync()) {                                  \
            cudaError_t e2__ = cudaStreamSynchronize(stream);        \
            if (e2__ != cudaSuccess)                                 \
                throw ::ihtb::Error(IHTB_ECUDA, std::string("kernel " #kernel " failed: ") + cudaGetErrorString(e2__)); \
        }                                                            \
    } while (0)

template <typename F>
static inline int32_t guard(F&& f) {
    try {
        f();
        return IHTB_OK;
    } catch (const Error& e) {
        set_last_error(e.what());
        return e.code;
    } catch (const std::bad_alloc&) {
        set_last_error("out of host memory");
        return IHTB_ENOMEM;
    } catch (const std::exception& e) {
        set_last_error(e.what());
        return IHTB_EINVAL;
    }
}

// ---- device buffer RAII --------------------------------------------------------------------
template <typename T>
struct DBuf {
    T* p = nullptr;
    size_t n = 0;
    DBuf() = default;
    explicit DBuf(size_t count) { alloc(count); }
    DBuf(const DBuf&) = delete;
    DBuf& operator=(const DBuf&) = delete;
    ~DBuf() { release(); }
    void alloc(size_t count) {
        release();
        n = count;
        if (count) {
            cudaError_t e = cudaMalloc((void**)&p, count * sizeof(T));
            if (e != cudaSuccess) {
                p = nullptr; n = 0;
                throw Error(IHTB_ENOMEM, std::string("cudaMalloc of ") + std::to_string(count * sizeof(T)) +
                                             " bytes failed: " + cudaGetErrorString(e));
            }
        }
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr; n = 0;
    }
    void zero(cudaStream_t s) { if (n) IHTB_CUDA(cudaMemsetAsync(p, 0, n * sizeof(T), s)); }
};

// pinned host buffer for scalar read-backs
template <typename T>
struct HBuf {
    T* p = nullptr;
    size_t n = 0;
    HBuf() = default;
    HBuf(const HBuf&) = delete;
    HBuf& operator=(const HBuf&) = delete;
    ~HBuf() { if (p) cudaFreeHost(p); }
    void alloc(size_t count) {
        if (p) cudaFreeHost(p);
        p = nullptr; n = count;
        if (count) IHTB_CUDA(cudaMallocHost((void**)&p, count * sizeof(T)));
    }
};

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device property of a kernel: set it once per (kernel, device),
// safely from several host threads (multi-device handles run one host thread per device).  geno.cu keeps the registry.
bool smem_attr_needed(const void* kernel, int device);
template <typename K>
static inline void ensure_dynamic_smem(K kernel, int bytes) {
    int dev = 0;
    IHTB_CUDA(cudaGetDevice(&dev));
    if (!smem_attr_needed(reinterpret_cast<const void*>(kernel), dev)) return;
    IHTB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
}

// ---- genotype handle -----------------------------------------------------------------------
struct TopkFuse;
// dense.cu (DENSE handles).  The dense X'v is the plain product sum_i x_ij v_i: no centring, the mean of v is not read.
ihtb_geno* dense_new_handle(int64_t n, int64_t p, int dtype, int standardize, int32_t den = 0);
void dense_upload(ihtb_geno* g, const void* x, int64_t ld_host, int64_t j_dst, int64_t ncols);
void dense_finalize(ihtb_geno* g);       // statistics / standardization, error-bound scale; IHTB_EDOMAIN on bad entries
int64_t dense_stream_bytes(const ihtb_geno* g);
void dense_decode_block(const ihtb_geno* g, int64_t i0, int64_t i1, int64_t j0, int64_t j1, double* d_out);
void dense_xt_v(const ihtb_geno* g, const double* dV, int64_t m, double* dOut, cudaStream_t s, DBuf<double>* part,
                const TopkFuse* tf);
void dense_sweep_kernel_only(const ihtb_geno* g, const double* dV, DBuf<double>* part, cudaStream_t s);
void dense_x_support(const ihtb_geno* g, const int64_t* d_idx, int64_t k, const double* d_coef, int64_t m,
                     double* d_out, cudaStream_t s);
void dense_xt_gather2(const ihtb_geno* g, const int64_t* d_cols_a, int64_t n_a, const int64_t* d_cols_b, int64_t n_b,
                      const double* d_v, int64_t m, double* d_out, cudaStream_t s);
// sum_i w_i x_ij, sum_i w_i x_ij^2, sum_i wy_i x_ij per column (init_beta), three p-vectors
void dense_init_beta_moments(const ihtb_geno* g, const double* d_w, const double* d_wy, double* d_sx, double* d_sxx,
                             double* d_sxy, cudaStream_t s);
// out[c*n + i] = x[i, cols[c]] in FP64 (cols[c] < 0: zeros)
void dense_decode_cols(const ihtb_geno* g, const int64_t* d_cols, int64_t k, double* d_out, cudaStream_t s);
// per-column scale and coefficient of the error bound of a sweep whose candidates are re-scored exactly:
// |df_j - exact_j| <= coef * scale_j * (sum|r| + |sum r|).  PLINK: the handle's sinv and the sweep mode's coefficient.
const double* geno_bound_scale(const ihtb_geno* g);
double geno_bound_coef(const ihtb_geno* g, double plink_coef);

}  // namespace ihtb

// A handle holds one of two matrix kinds.  PLINK: the 2-bit packed genotypes below.  DENSE: an n x p matrix of FP64 or
// FP32 entries (dense.cu), column-major with a padded leading dimension; the fit, CV and debias code reads it through
// the dispatch points that test `kind`.
enum { GENO_PLINK = 0, GENO_DENSE = 1 };

struct ihtb_geno {
    int kind = 0;             // GENO_PLINK | GENO_DENSE
    int device = 0;
    int64_t n = 0;            // samples
    int64_t p = 0;            // local SNP columns
    int64_t j0 = 0;           // global index of local column 0 (SNP-sharded fits)
    int64_t nbytes = 0;       // ceil(n/4)
    int64_t stride = 0;       // padded bytes per column: multiple of 128 (= 512-sample slabs), zero padded
    // Quad-interleaved slab-major tiles: the samples are cut into slabs of 512 (128 bytes per column), one slab of all
    // columns is contiguous, and inside a slab columns are grouped by four with the 32-bit words of their four 128-byte
    // chunks interleaved, so that 16 consecutive bytes hold word w of columns 4q..4q+3.  Byte b of column j lives at
    //   bed + (b>>7)*cs_s + (j>>2)*512 + ((b&127)>>2)*16 + (j&3)*4 + (b&3),  cs_s = p4*128.
    // A sweep stage of 128 columns is then one contiguous 16 KB bulk copy, and one 128-bit shared-memory load per lane
    // feeds four columns with lane = word position, which is what the table lookups of the sweeps need (sweep_lut.cu).
    int64_t cs_s = 0;         // bytes per slab
    int64_t p4 = 0;           // columns allocated per slab (p rounded up to a multiple of 4; padding columns are zero)
    int center = 1, scale = 1, impute = 1;
    int sm_count = 148;
    ihtb::DBuf<uint8_t> bed;  // p * stride bytes
    // Ternary copy for the table sweeps (sweep_lut.cu), built at finalize when memory allows (geno.cu build_tern):
    // the same quad-interleaved tiles, but a byte holds FIVE dosages in base 3 (d0 + 3 d1 + 9 d2 + 27 d3 + 81 d4 <= 242;
    // missing -> 0 like the 2-bit sweep, the CSR correction of the epilogue is unchanged), so a 128-byte chunk covers 640
    // samples instead of 512: 20 % fewer bytes from HBM AND 20 % fewer table lookups per genotype.  Lossless: every other
    // kernel keeps reading the PLINK codes in `bed`.
    ihtb::DBuf<uint8_t> tern;         // tern_slabs * p4 * 128 bytes (empty: the sweeps read `bed`)
    int64_t tern_slabs = 0;           // ceil(n / 640)
    ihtb::DBuf<double> mu, sinv;
    // sgn_j = sinv_j * max(sqrt(sum_i g_ij^2), 1): per-column scale of the L2 error bounds of the table sweeps --
    // the absolute dot product sum_i g_ij |u_i| that every rounding error is relative to is at most
    // sqrt(sum_i g_ij^2) * ||u||_2 (Cauchy-Schwarz), which is far tighter than 2 ||u||_1 for the PAIR sweep
    ihtb::DBuf<double> sgn;
    ihtb::DBuf<int32_t> nmiss;
    // CSR of missing samples per column (sparse imputation correction of the sweep; PLINK and standardized FIX16 handles)
    ihtb::DBuf<int64_t> miss_ptr;   // [p+1]
    ihtb::DBuf<int32_t> miss_idx;   // sample indices
    int64_t total_missing = 0;
    bool ready = false;             // columns loaded and statistics computed (false between create_empty and finalize)
    // ---- DENSE handles (dense.cu) ----
    int dtype = 0;                  // IHTB_DENSE_F64 | IHTB_DENSE_F32 | IHTB_DENSE_FIX16
    int standardize = 0;            // 1: standardize_genotypes! applied at finalize (NaN / the missing code = missing)
    int32_t den = 0;                // FIX16: code c stands for c / den (1..65534); 0 for float storage
    int64_t ld = 0;                 // device leading dimension in elements: n rounded up to a whole number of sweep slabs
    ihtb::DBuf<uint8_t> dense;      // p * ld elements, zero padded below row n
    // per-column error-bound scale: max_i |x_ij| of the stored (standardized) matrix; FIX16 dense_finalize
    ihtb::DBuf<double> dscale;
    double dcoef = 0.0;             // error-bound coefficient of the dense sweep + re-scoring (dense_bound_coef)
    // staging buffers and streams of ihtb_geno_load_bgen_columns (bgen.cu), kept between its calls so that pinned memory
    // is allocated once per load rather than once per batch; released at finalize
    std::shared_ptr<void> bgen_stage;
};
static inline bool geno_is_dense(const ihtb_geno* g) { return g->kind == GENO_DENSE; }

static inline void geno_require_ready(const ihtb_geno* g) {
    IHTB_CHECK(g && g->ready, IHTB_EINVAL, "genotype handle is not finalized (ihtb_geno_finalize)");
}

// what kernels see of a genotype handle
struct GenoView {
    const uint8_t* bed;
    int64_t cs_s, nbytes, stride, n, p;
    const double* mu;
    const double* sinv;
    const int32_t* nmiss;
    int impute;
};
static inline GenoView geno_view(const ihtb_geno* g) {
    return GenoView{g->bed.p, g->cs_s, g->nbytes, g->stride, g->n, g->p, g->mu.p, g->sinv.p, g->nmiss.p, g->impute};
}
// address of byte b of column j (ihtb_geno::bed); the 4 bytes of a 32-bit word (4-byte aligned b) are contiguous
__device__ __forceinline__ const uint8_t* gv_ptr(const GenoView& g, int64_t j, int64_t b) {
    return g.bed + (b >> 7) * g.cs_s + (j >> 2) * 512 + ((b & 127) >> 2) * 16 + (j & 3) * 4 + (b & 3);
}

namespace ihtb {

// ---- device helpers --------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Deterministic block reduction (fixed tree); result valid in thread 0. `sh` needs 32 doubles.
__device__ __forceinline__ double block_sum(double v, double* sh) {
    v = warp_sum(v);
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) sh[w] = v;
    __syncthreads();
    int nw = (blockDim.x + 31) >> 5;
    v = (threadIdx.x < nw) ? sh[threadIdx.x] : 0.0;
    if (w == 0) v = warp_sum(v);
    return v;
}

// ---- kernels implemented in other translation units -------------------------------------------
// sweep.cu
void sweep_xt_v(const ihtb_geno* g, const double* dV, int64_t m, double* dOut, int mode, cudaStream_t s,
                double* sweep_seconds);
// support.cu
void x_support(const ihtb_geno* g, const int64_t* d_idx_local, int64_t k, const double* d_coef, int64_t m,
               double* d_out, cudaStream_t s);
void xt_gather(const ihtb_geno* g, const int64_t* d_cols_local, int64_t ncols, const double* d_v, int64_t m,
               const double* d_vsum /*[m] device*/, double* d_out /*[ncols*m]*/, cudaStream_t s);
// m = 1 takes the nibble-table kernel whatever the list length (a column's value never depends on the list); `blocked`
// is kept for source compatibility and ignored
void xt_gather2(const ihtb_geno* g, const int64_t* d_cols_a, int64_t n_a, const int64_t* d_cols_b, int64_t n_b,
                const double* d_v, int64_t m, const double* d_vsum, double* d_out, cudaStream_t s, bool blocked = false);

struct TopkFuse;
// dense.cu (DENSE handles).  The dense X'v is the plain product sum_i x_ij v_i: no centring, d_vbar is not read.
void dense_xt_v(const ihtb_geno* g, const double* dV, int64_t m, double* dOut, cudaStream_t s, void* scratch_any,
                const TopkFuse* tf);
void dense_x_support(const ihtb_geno* g, const int64_t* d_idx, int64_t k, const double* d_coef, int64_t m,
                     double* d_out, cudaStream_t s);
void dense_xt_gather2(const ihtb_geno* g, const int64_t* d_cols_a, int64_t n_a, const int64_t* d_cols_b, int64_t n_b,
                      const double* d_v, int64_t m, double* d_out, cudaStream_t s);
// Sum_i w_i x_ij, Sum_i w_i x_ij^2, Sum_i wy_i x_ij per column (init_beta), three p-vectors
void dense_init_beta_moments(const ihtb_geno* g, const double* d_w, const double* d_wy, double* d_sx, double* d_sxx,
                             double* d_sxy, cudaStream_t s, void* scratch_any);
// out[c*n + i] = x[i, cols[c]] in FP64 (cols[c] < 0: zeros)
void dense_decode_cols(const ihtb_geno* g, const int64_t* d_cols, int64_t k, double* d_out, cudaStream_t s);
// per-column scale and coefficient of the error bound of a sweep whose candidates are re-scored exactly
// (|df_j - exact_j| <= coef * scale_j * (sum|r| + |sum r|)); PLINK: the handle's sinv with the sweep mode's coefficient
const double* geno_bound_scale(const ihtb_geno* g);
double geno_bound_coef(const ihtb_geno* g, double plink_coef);

}  // namespace ihtb
