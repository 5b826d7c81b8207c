// The dominant kernel: transpose matvec X'v over the 2-bit packed matrix.
// Replaces mul!(v.df, Transpose(x), v.r) (reference src/utilities.jl:133, executed inside SnpArrays.jl) and the
// skinny multi-RHS SnpArrays.mul!(v.p_by_r, Transpose(sla), v.n_by_r) (src/multivariate.jl:85).
//
// All variants compute, per column j and right-hand side t, with u = v - mean(v):
//     A_jt = sum_{observed i} dosage_ij * u_it            (dense pass over the packed bytes; code 01 counts 0)
// and an epilogue adds the sparse mean-imputation term and scales:
//     out_jt = sinv_j * (A_jt + mu_j * sum_{missing i} u_it)
// which equals sinv_j * (sum_i gimp_ij v_it - mu_j sum_i v_it) because mean imputation keeps sum_i gimp_ij = n mu_j.
//
//  EXACT: FP64 nibble-indexed lookup tables in shared memory, slab partials in FP64 (sweep_lut64.cu).
//  FAST : FP32 byte-indexed lookup tables in shared memory (sweep_lut.cu).
#include "common.cuh"
#include "pairer.cuh"
#include "topk.cuh"

namespace ihtb {

void sweep_fast_partials(const ihtb_geno* g, const double* d_v, const double* d_vbar, float* d_part, int64_t* n_slabs,
                         cudaStream_t s);
int64_t sweep_fast_num_slabs(const ihtb_geno* g);
void sweep_exact_lut_partials(const ihtb_geno* g, const double* d_v, const double* d_vbar, double* d_part, cudaStream_t s,
                              int cls = 0);
void sweep_pair_partials(const ihtb_geno* g, const double* d_v0, const double* d_v1, const double* d_vbar,
                         const float* d_scale, float* d_part, cudaStream_t s);

// out_j = sinv_j * (sum_s part[s][j] + mu_j * (impute ? sum_{i in miss_j} u_i : -vbar * nmiss_j))
// tf (optional, tf.keyL != NULL): the first stage of the candidate selection that follows a univariate sweep (topk.cuh
// TopkFuse) -- keys of |df_j| with the sweep's error bound and the first digit histogram -- computed here, where df_j is
// produced, instead of in a kernel of its own.  256 threads per CTA.
template <typename T>
__global__ void __launch_bounds__(256)
k_sweep_epilogue(const T* __restrict__ part, int64_t n_slabs, int64_t p,
                 const double* __restrict__ mu, const double* __restrict__ sinv,
                 const int32_t* __restrict__ nmiss, const int64_t* __restrict__ miss_ptr,
                 const int32_t* __restrict__ miss_idx, const double* __restrict__ v,
                 const double* __restrict__ vbar_p,
                 int impute, double* __restrict__ out, const float* __restrict__ scale_p = nullptr,
                 TopkFuse tf = TopkFuse()) {
    __shared__ int sh[TOPK_BINS];
    const bool fuse = tf.keyL != nullptr;
    if (fuse) {
        topk_first_kernel_housekeeping(tf.hist_other, tf.st, tf.cand, tf.cand_fill);
        for (int b = threadIdx.x; b < TOPK_BINS; b += blockDim.x) sh[b] = 0;
        __syncthreads();
    }
    int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (j < p) {
        const double vbar = *vbar_p;
        double a = 0.0;
        for (int64_t s = 0; s < n_slabs; ++s) a += (double)part[s * p + j];
        if (scale_p) a /= (double)*scale_p;            // pair sweep: sums of 2^e-scaled values (exact division)
        double corr = 0.0;
        int nm = nmiss[j];
        if (nm) {
            if (impute) {
                for (int64_t e = miss_ptr[j]; e < miss_ptr[j + 1]; ++e) corr += v[miss_idx[e]] - vbar;
            } else {
                corr = -vbar * (double)nm;
            }
        }
        const double df = sinv[j] * (a + mu[j] * corr);
        out[j] = df;
        if (fuse) {
            // k_keys_hist0's arithmetic for b0 = 0, eta = 1: bound = coef * (sum |r| + |sum r|) from the score sums
            const double bound = tf.bound_coef * (tf.scal[1] + fabs(tf.scal[0]));
            const double w = tf.wt ? tf.wt[j] : 1.0;
            uint32_t kl, ku;
            topk_make_keys(0.0 + 1.0 * df, w, fabs(1.0) * tf.scale[j] * bound * w, kl, ku);
            tf.keyL[j] = kl; tf.keyU[j] = ku;
            atomicAdd(&sh[kl >> 21], 1);
        }
    }
    if (fuse) {
        __syncthreads();
        for (int b = threadIdx.x; b < TOPK_BINS; b += blockDim.x)
            if (sh[b]) atomicAdd(&tf.hist[b], sh[b]);
    }
}

__global__ void k_vec_mean(const double* __restrict__ v, int64_t n, double* __restrict__ out) {
    // single block, fixed order: mean of a right-hand side (only used by the stand-alone ihtb_xt_v entry point)
    __shared__ double sh[32];
    double a = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) a += v[i];
    a = block_sum(a, sh);
    if (threadIdx.x == 0) out[0] = a / (double)n;
}

// pair sweep prelude: power-of-two scales that bring max |v - mean| of each right-hand side below 2^9 (the half2 tables
// of k_sweep_ldg<.., true> then cannot overflow: entries <= 8 * 2^9, sums of four <= 2^14)
__global__ void k_pair_scale(const double* __restrict__ v0, const double* __restrict__ v1, int64_t n,
                             const double* __restrict__ vbar, float* __restrict__ scale) {
    __shared__ double sh[32];
    for (int t = 0; t < 2; ++t) {
        const double* v = t ? v1 : v0;
        const double vb = vbar[t];
        double m = 0.0;
        for (int64_t i = threadIdx.x; i < n; i += blockDim.x) m = fmax(m, fabs(v[i] - vb));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
        __syncthreads();
        if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = m;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < (int)(blockDim.x >> 5); ++w) m = fmax(m, sh[w]);
            int e = 0;
            if (m > 0.0 && isfinite(m)) frexp(m, &e);        // m = f * 2^e, f in [0.5, 1)  ->  m < 2^e
            scale[t] = ldexpf(1.0f, 9 - e);
        }
    }
}

// ||v - mean||_2 in FP64, one block, fixed order (the L2 error bounds of the PAIR sweep)
__global__ void k_l2norm(const double* __restrict__ v, int64_t n, const double* __restrict__ vbar, double* __restrict__ out) {
    __shared__ double sh[32];
    const double vb = vbar[0];
    double a = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) { const double u = v[i] - vb; a += u * u; }
    a = block_sum(a, sh);
    if (threadIdx.x == 0) out[0] = sqrt(a);
}

struct SweepScratch {
    DBuf<double> part64;
    DBuf<float> part32;
    DBuf<float> scale;
};

// dV: n x m column-major device array; dOut: p x m. d_vbar[t] = mean of column t (DEVICE array, so a sweep can be
// enqueued right behind the kernel that produced the mean without a host round trip).
// d_l2 (optional, m doubles, PAIR mode): ||v_t - mean||_2 of every right-hand side, for the L2 error bounds.
// tf (optional, single right-hand side): first stage of the |df| selection, run by the epilogue (topk.cuh TopkFuse).
void sweep_xt_v_with_means(const ihtb_geno* g, const double* dV, const double* d_vbar, int64_t m, double* dOut,
                           int mode, cudaStream_t s, void* scratch_any, float* sweep_ms, double* d_l2 = nullptr,
                           const TopkFuse* tf = nullptr) {
    IHTB_CHECK(!tf || (m == 1 && mode != IHTB_SWEEP_PAIR), IHTB_EINVAL, "fused selection stage: one right-hand side");
    const TopkFuse fuse = tf ? *tf : TopkFuse();
    SweepScratch local;
    SweepScratch* sc = scratch_any ? reinterpret_cast<SweepScratch*>(scratch_any) : &local;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (sweep_ms) {
        IHTB_CUDA(cudaEventCreate(&e0)); IHTB_CUDA(cudaEventCreate(&e1));
        IHTB_CUDA(cudaEventRecord(e0, s));
    }
    if (geno_is_dense(g)) {
        // every mode computes the same exact FP64 product (dense.cu); a dense handle never pairs (d_l2 stays unused)
        dense_xt_v(g, dV, m, dOut, s, &sc->part64, tf);
    } else {
        if (d_l2)
            for (int64_t t = 0; t < m; ++t) IHTB_LAUNCH(k_l2norm, 1, 1024, 0, s, dV + t * g->n, g->n, d_vbar + t, d_l2 + t);
        for (int64_t t = 0; t < m; ++t) {
            const double* v = dV + t * g->n;
            double* out = dOut + t * g->p;
            if (mode == IHTB_SWEEP_PAIR && t + 1 < m) {
                // two right-hand sides per pass over the matrix (half2 tables); an odd last one takes the FAST path below
                const int64_t n_slabs = sweep_fast_num_slabs(g);
                if (sc->part32.n < (size_t)(2 * n_slabs * g->p)) sc->part32.alloc((size_t)(2 * n_slabs * g->p));
                if (sc->scale.n < 2) sc->scale.alloc(2);
                IHTB_LAUNCH(k_pair_scale, 1, 1024, 0, s, v, v + g->n, g->n, d_vbar + t, sc->scale.p);
                sweep_pair_partials(g, v, v + g->n, d_vbar + t, sc->scale.p, sc->part32.p, s);
                for (int h = 0; h < 2; ++h)
                    IHTB_LAUNCH((k_sweep_epilogue<float>), (unsigned)ceil_div(g->p, 256), 256, 0, s,
                                sc->part32.p + (size_t)h * n_slabs * g->p, n_slabs, g->p, g->mu.p, g->sinv.p, g->nmiss.p,
                                g->miss_ptr.p, g->miss_idx.p, v + h * g->n, d_vbar + t + h, g->impute, out + h * g->p,
                                sc->scale.p + h);
                ++t;
                continue;
            }
            if (mode == IHTB_SWEEP_EXACT) {
                const int64_t n_slabs = g->stride / 128;
                if (sc->part64.n < (size_t)(n_slabs * g->p)) sc->part64.alloc((size_t)(n_slabs * g->p));
                sweep_exact_lut_partials(g, v, d_vbar + t, sc->part64.p, s);
                IHTB_LAUNCH((k_sweep_epilogue<double>), (unsigned)ceil_div(g->p, 256), 256, 0, s, sc->part64.p, n_slabs,
                            g->p, g->mu.p, g->sinv.p, g->nmiss.p, g->miss_ptr.p, g->miss_idx.p, v, d_vbar + t,
                            g->impute, out, (const float*)nullptr, fuse);
            } else {
                int64_t n_slabs = sweep_fast_num_slabs(g);
                if (sc->part32.n < (size_t)(n_slabs * g->p)) sc->part32.alloc((size_t)(n_slabs * g->p));
                sweep_fast_partials(g, v, d_vbar + t, sc->part32.p, &n_slabs, s);
                IHTB_LAUNCH((k_sweep_epilogue<float>), (unsigned)ceil_div(g->p, 256), 256, 0, s, sc->part32.p, n_slabs,
                            g->p, g->mu.p, g->sinv.p, g->nmiss.p, g->miss_ptr.p, g->miss_idx.p, v, d_vbar + t,
                            g->impute, out, (const float*)nullptr, fuse);
            }
        }
    }
    if (sweep_ms) {
        IHTB_CUDA(cudaEventRecord(e1, s));
        IHTB_CUDA(cudaEventSynchronize(e1));
        IHTB_CUDA(cudaEventElapsedTime(sweep_ms, e0, e1));
        cudaEventDestroy(e0); cudaEventDestroy(e1);
    }
}

// ---- lock-step pairing of two fits' sweeps (pairer.cuh) -------------------------------------------------------------
__global__ void k_copy2(const double* __restrict__ a, const double* __restrict__ b, double* __restrict__ out) {
    out[0] = a[0]; out[1] = b[0];
}

SweepPairer::SweepPairer(int dev) : device(dev) {
    IHTB_CUDA(cudaSetDevice(dev));
    for (int i = 0; i < 2; ++i) IHTB_CUDA(cudaEventCreateWithFlags(&ready[i], cudaEventDisableTiming));
    IHTB_CUDA(cudaEventCreateWithFlags(&done, cudaEventDisableTiming));
    IHTB_CUDA(cudaMalloc((void**)&d_vbar2, 2 * sizeof(double)));
    IHTB_CUDA(cudaMalloc((void**)&d_l2, 2 * sizeof(double)));
    scratch = new SweepScratch();
}
SweepPairer::~SweepPairer() {
    cudaSetDevice(device);
    cudaDeviceSynchronize();
    for (int i = 0; i < 2; ++i) if (ready[i]) cudaEventDestroy(ready[i]);
    if (done) cudaEventDestroy(done);
    if (d_vbar2) cudaFree(d_vbar2);
    if (d_l2) cudaFree(d_l2);
    delete reinterpret_cast<SweepScratch*>(scratch);
}

void SweepPairer::leave() {
    std::lock_guard<std::mutex> lk(mu);
    --active;
    cv.notify_all();
}

bool SweepPairer::sweep(int slot, const ihtb_geno* g, const double* d_v, const double* d_vbar, double* d_out,
                        cudaStream_t s, void* solo_scratch) {
    const int other = slot ^ 1;
    IHTB_CUDA(cudaEventRecord(ready[slot], s));        // v / vbar of this fit are complete at this point of its stream
    std::unique_lock<std::mutex> lk(mu);
    if (active >= 2 && !geno_is_dense(g)) {
        req[slot] = Req{d_v, d_vbar, d_out, s};
        has[slot] = true;
        if (has[other]) {
            // second to arrive: launch one pass for both on this stream, behind the partner's producer kernels
            const Req a = req[0], b = req[1];
            SweepScratch* sc = reinterpret_cast<SweepScratch*>(scratch);
            const int64_t n_slabs = sweep_fast_num_slabs(g);
            if (sc->part32.n < (size_t)(2 * n_slabs * g->p)) sc->part32.alloc((size_t)(2 * n_slabs * g->p));
            if (sc->scale.n < 2) sc->scale.alloc(2);
            IHTB_CUDA(cudaStreamWaitEvent(s, ready[other], 0));
            IHTB_LAUNCH(k_copy2, 1, 1, 0, s, a.vbar, b.vbar, d_vbar2);
            IHTB_LAUNCH(k_pair_scale, 1, 1024, 0, s, a.v, b.v, g->n, d_vbar2, sc->scale.p);
            IHTB_LAUNCH(k_l2norm, 1, 1024, 0, s, a.v, g->n, d_vbar2, d_l2);
            IHTB_LAUNCH(k_l2norm, 1, 1024, 0, s, b.v, g->n, d_vbar2 + 1, d_l2 + 1);
            sweep_pair_partials(g, a.v, b.v, d_vbar2, sc->scale.p, sc->part32.p, s);
            const Req* rq[2] = {&a, &b};
            for (int h = 0; h < 2; ++h)
                IHTB_LAUNCH((k_sweep_epilogue<float>), (unsigned)ceil_div(g->p, 256), 256, 0, s,
                            sc->part32.p + (size_t)h * n_slabs * g->p, n_slabs, g->p, g->mu.p, g->sinv.p, g->nmiss.p,
                            g->miss_ptr.p, g->miss_idx.p, rq[h]->v, d_vbar2 + h, g->impute, rq[h]->out, sc->scale.p + h);
            IHTB_CUDA(cudaEventRecord(done, s));
            has[0] = has[1] = false;
            ++round;
            ++n_pair;
            cv.notify_all();
            return true;
        }
        // first to arrive: wait for the partner's sweep (or for its departure)
        const unsigned long long r0 = round;
        cv.wait(lk, [&] { return round != r0 || active < 2; });
        if (round != r0) {
            IHTB_CUDA(cudaStreamWaitEvent(s, done, 0));    // the leader's stream wrote this fit's df
            return true;
        }
        has[slot] = false;                                 // partner left: sweep alone
    }
    ++n_solo;
    lk.unlock();
    sweep_xt_v_with_means(g, d_v, d_vbar, 1, d_out, IHTB_SWEEP_FAST, s, solo_scratch, nullptr, nullptr);
    return false;
}

void* sweep_scratch_create() { return new SweepScratch(); }
void sweep_scratch_destroy(void* p) { delete reinterpret_cast<SweepScratch*>(p); }

}  // namespace ihtb

using namespace ihtb;

extern "C" int32_t ihtb_xt_v(const ihtb_geno* g, const double* V, int64_t m, double* out, int32_t sweep_mode) {
    return guard([&] {
        IHTB_CHECK(g && V && out && m >= 1, IHTB_EINVAL, "bad argument");
        geno_require_ready(g);
        IHTB_CHECK(sweep_mode == IHTB_SWEEP_FAST || sweep_mode == IHTB_SWEEP_EXACT || sweep_mode == IHTB_SWEEP_PAIR,
                   IHTB_EINVAL, "bad sweep_mode");
        IHTB_CUDA(cudaSetDevice(g->device));
        DBuf<double> dV((size_t)(g->n * m)), dOut((size_t)(g->p * m)), dmean((size_t)m);
        IHTB_CUDA(cudaMemcpy(dV.p, V, g->n * m * sizeof(double), cudaMemcpyHostToDevice));
        for (int64_t t = 0; t < m; ++t)
            IHTB_LAUNCH(k_vec_mean, 1, 1024, 0, 0, dV.p + t * g->n, g->n, dmean.p + t);
        sweep_xt_v_with_means(g, dV.p, dmean.p, m, dOut.p, sweep_mode, 0, nullptr, nullptr, nullptr);
        IHTB_CUDA(cudaMemcpy(out, dOut.p, g->p * m * sizeof(double), cudaMemcpyDeviceToHost));
    });
}

// ---- measurement hooks (bench.py): sweep timed alone on a device-resident vector, CUDA events on its stream ------
namespace ihtb {
void sweep_fast_kernel_only(const ihtb_geno* g, const double* d_v, const double* d_vbar, float* d_part, cudaStream_t s);
__global__ void k_fill_vec(double* v, int64_t n, uint64_t seed) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t x = seed + (uint64_t)i * 0x9E3779B97F4A7C15ull;
    x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 27; x *= 0x94D049BB133111EBull; x ^= x >> 31;
    v[i] = ((double)(x >> 11) * (1.0 / 9007199254740992.0) - 0.5) * 2.0;
}
}  // namespace ihtb

extern "C" int32_t ihtb_sweep_bench(const ihtb_geno* g, int32_t sweep_mode, int32_t warmup, int32_t reps,
                                    double* ms_kernel, double* ms_total) {
    return guard([&] {
        IHTB_CHECK(g && reps >= 1 && warmup >= 0, IHTB_EINVAL, "bad argument");
        geno_require_ready(g);
        IHTB_CUDA(cudaSetDevice(g->device));
        cudaStream_t s;
        IHTB_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
        const int64_t mrhs = sweep_mode == IHTB_SWEEP_PAIR ? 2 : 1;       // PAIR: two right-hand sides per launch
        DBuf<double> dV((size_t)(g->n * mrhs)), dOut((size_t)(g->p * mrhs));
        IHTB_LAUNCH(k_fill_vec, (unsigned)ceil_div(g->n * mrhs, 256), 256, 0, s, dV.p, g->n * mrhs, 12345ull);
        DBuf<double> dmean((size_t)mrhs);
        for (int64_t t = 0; t < mrhs; ++t) IHTB_LAUNCH(k_vec_mean, 1, 1024, 0, s, dV.p + t * g->n, g->n, dmean.p + t);
        SweepScratch sc;
        cudaEvent_t e0, e1;
        IHTB_CUDA(cudaEventCreate(&e0)); IHTB_CUDA(cudaEventCreate(&e1));
        // milliseconds per call of `launch`, by CUDA events around `reps` calls on s
        auto time_reps = [&](auto&& launch) {
            IHTB_CUDA(cudaEventRecord(e0, s));
            for (int i = 0; i < reps; ++i) launch();
            IHTB_CUDA(cudaEventRecord(e1, s));
            IHTB_CUDA(cudaEventSynchronize(e1));
            float ms = 0.f;
            IHTB_CUDA(cudaEventElapsedTime(&ms, e0, e1));
            return (double)(ms / reps);
        };
        for (int i = 0; i < warmup; ++i)
            sweep_xt_v_with_means(g, dV.p, dmean.p, mrhs, dOut.p, sweep_mode, s, &sc, nullptr, nullptr);
        // (a) whole sweep = partial-sum kernel + epilogue
        const double total = time_reps([&] {
            sweep_xt_v_with_means(g, dV.p, dmean.p, mrhs, dOut.p, sweep_mode, s, &sc, nullptr, nullptr);
        });
        if (ms_total) *ms_total = total;
        // (b) the dominant kernel alone
        if (ms_kernel) {
            *ms_kernel = 0.0;
            if (geno_is_dense(g))
                *ms_kernel = time_reps([&] { dense_sweep_kernel_only(g, dV.p, &sc.part64, s); });
            else if (sweep_mode == IHTB_SWEEP_PAIR)
                *ms_kernel = time_reps([&] {
                    sweep_pair_partials(g, dV.p, dV.p + g->n, dmean.p, sc.scale.p, sc.part32.p, s);
                });
            else if (sweep_mode == IHTB_SWEEP_FAST)
                *ms_kernel = time_reps([&] { sweep_fast_kernel_only(g, dV.p, dmean.p, sc.part32.p, s); });
            else
                *ms_kernel = time_reps([&] { sweep_exact_lut_partials(g, dV.p, dmean.p, sc.part64.p, s); });
        }
        cudaEventDestroy(e0); cudaEventDestroy(e1);
        cudaStreamDestroy(s);
    });
}

// ---- class sums for init_beta (reference initialize_beta!, src/utilities.jl:776-812) -------------------------------
// W1_j = sum_i v_i [g_ij = 1], W2_j = sum_i v_i [g_ij = 2], Wm_j = sum_i v_i [g_ij missing]  (v NOT centred).
// With the four possible standardised values of a column, sum x, sum x^2 and sum x*y over the training samples follow
// from these sums for v = w and v = w.*y, so the univariate regressions need two exact passes over the matrix.
namespace ihtb {

__global__ void k_class_epilogue(const double* __restrict__ part1, const double* __restrict__ part2, int64_t n_slabs,
                                 int64_t p, const int64_t* __restrict__ miss_ptr, const int32_t* __restrict__ miss_idx,
                                 const double* __restrict__ v, double* __restrict__ out1, double* __restrict__ out2,
                                 double* __restrict__ outm) {
    int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (j >= p) return;
    double a = 0.0, b = 0.0, m = 0.0;
    for (int64_t s = 0; s < n_slabs; ++s) { a += part1[s * p + j]; b += part2[s * p + j]; }
    for (int64_t e = miss_ptr[j]; e < miss_ptr[j + 1]; ++e) m += v[miss_idx[e]];
    out1[j] = a; out2[j] = b; outm[j] = m;
}

void sweep_class_sums(const ihtb_geno* g, const double* d_v, double* d_w1, double* d_w2, double* d_wm, cudaStream_t s,
                      void* scratch_any) {
    SweepScratch* sc = reinterpret_cast<SweepScratch*>(scratch_any);
    // the table-driven FP64 sweep (sweep_lut64.cu) with the indicator maps instead of the dosage, one pass per class
    const int64_t ns = g->stride / 128;
    if (sc->part64.n < (size_t)(2 * ns * g->p)) sc->part64.alloc((size_t)(2 * ns * g->p));
    double* q1 = sc->part64.p;
    double* q2 = sc->part64.p + ns * g->p;
    sweep_exact_lut_partials(g, d_v, nullptr, q1, s, 1);
    sweep_exact_lut_partials(g, d_v, nullptr, q2, s, 2);
    IHTB_LAUNCH(k_class_epilogue, (unsigned)ceil_div(g->p, 256), 256, 0, s, q1, q2, ns, g->p, g->miss_ptr.p,
                g->miss_idx.p, d_v, d_w1, d_w2, d_wm);
}

}  // namespace ihtb
