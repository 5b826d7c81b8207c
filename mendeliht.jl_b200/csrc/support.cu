// Support-only kernels: x[:, idx] * coef (gather matvec) and exact FP64 column dots x[:, cols]' * V.
// Replace the getindex loops of the reference: update_xb! (src/utilities.jl:95-111), iht_stepsize!
// (src/utilities.jl:728-743) and their multivariate forms (src/multivariate.jl:24,234); the column dots
// re-score top-k candidates exactly (same value mul!(df, Transpose(x), r) gives for those columns).
#include "common.cuh"
#include "comm.cuh"
#include <algorithm>
#include <memory>
#include <mutex>
#include <unordered_map>

namespace ihtb {

constexpr int XS_CHUNK = 32;  // columns staged per shared-memory table refill

// out[i, t] = sum_c x[i, idx_c] * coef[c, t], ascending c (the order the reference's single-thread loop uses).
// One thread per packed byte (4 samples). tab[c][code][t] = ((dos(code) - mu) * sinv) * coef[c, t].
// PUSH (M == 1, SNP-sharded fits): instead of `out`, the partial vector is stored into slot[parity][my_rank] of EVERY
// rank through the IPC-mapped peer pointers in `pv`, and the last CTA publishes the flags (comm.cuh) -- the all-reduce
// that follows is then a local sum of nranks slots (k_p2p_reduce).
template <int M, bool PUSH>
__global__ void __launch_bounds__(256)
k_x_support(GenoView gv, const int64_t* __restrict__ idx, int64_t k, const double* __restrict__ coef,
            double* __restrict__ out, P2PView pv, unsigned long long seq) {
    const int64_t nbytes = gv.nbytes, n = gv.n;
    const double* __restrict__ mu = gv.mu;
    const double* __restrict__ sinv = gv.sinv;
    const int impute = gv.impute;
    __shared__ double tab[XS_CHUNK][4][M];
    __shared__ int64_t cols[XS_CHUNK];
    int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    double acc[4][M];
#pragma unroll
    for (int s = 0; s < 4; ++s)
#pragma unroll
        for (int t = 0; t < M; ++t) acc[s][t] = 0.0;

    for (int64_t c0 = 0; c0 < k; c0 += XS_CHUNK) {
        int nc = (int)((k - c0 < XS_CHUNK) ? (k - c0) : XS_CHUNK);
        __syncthreads();
        for (int e = threadIdx.x; e < nc * 4 * M; e += blockDim.x) {
            int c = e / (4 * M), code = (e / M) & 3, t = e % M;
            int64_t j = idx[c0 + c];
            double m = mu[j];
            double g = (code == 2) ? 1.0 : (code == 3) ? 2.0 : (code == 1) ? (impute ? m : 0.0) : 0.0;
            double x = __dmul_rn(__dsub_rn(g, m), sinv[j]);
            tab[c][code][t] = __dmul_rn(x, coef[(c0 + c) + (int64_t)t * k]);
            if (code == 0 && t == 0) cols[c] = j;
        }
        __syncthreads();
        if (b < nbytes) {
            for (int c = 0; c < nc; ++c) {
                uint32_t byte = *gv_ptr(gv, cols[c], b);
#pragma unroll
                for (int s = 0; s < 4; ++s) {
                    uint32_t code = (byte >> (2 * s)) & 3u;
#pragma unroll
                    for (int t = 0; t < M; ++t) acc[s][t] = __dadd_rn(acc[s][t], tab[c][code][t]);
                }
            }
        }
    }
    if (PUSH) {
        // stage the CTA's 1024 contiguous samples so that every peer store is a full 16-byte lane of a 128-byte line
        // (NVLink write packets with all bytes enabled)
        __shared__ double stage[PUSH ? 1024 : 1];
        __syncthreads();
#pragma unroll
        for (int s = 0; s < 4; ++s) stage[4 * threadIdx.x + s] = acc[s][0];
        __syncthreads();
        const int64_t base = 1024 * (int64_t)blockIdx.x;
        for (int e = 2 * threadIdx.x; e < 1024; e += 512) {
            const int64_t i = base + e;
            if (i + 1 < n) {
                const double2 x = make_double2(stage[e], stage[e + 1]);
                for (int r = 0; r < pv.nranks; ++r) *reinterpret_cast<double2*>(pv.push_slot[r] + i) = x;
            } else if (i < n) {
                for (int r = 0; r < pv.nranks; ++r) pv.push_slot[r][i] = stage[e];
            }
        }
        p2p_publish(pv, seq);
        return;
    }
    if (b < nbytes) {
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            int64_t i = 4 * b + s;
            if (i < n)
#pragma unroll
                for (int t = 0; t < M; ++t) out[i + (int64_t)t * n] = acc[s][t];
        }
    }
}

template <int M>
static void launch_x_support(const ihtb_geno* g, const int64_t* d_idx, int64_t k, const double* d_coef, double* d_out,
                             cudaStream_t s) {
    IHTB_LAUNCH((k_x_support<M, false>), (unsigned)ceil_div(g->nbytes, 256), 256, 0, s, geno_view(g), d_idx, k, d_coef,
                d_out, P2PView{}, 0ull);
}

void x_support_push(const ihtb_geno* g, const int64_t* d_idx, int64_t k, const double* d_coef, ihtb_comm* c,
                    cudaStream_t s) {
    IHTB_LAUNCH((k_x_support<1, true>), (unsigned)ceil_div(g->nbytes, 256), 256, 0, s, geno_view(g), d_idx, k, d_coef,
                (double*)nullptr, p2p_view(c), (unsigned long long)(c->seq[0] + 1));
}

void x_support(const ihtb_geno* g, const int64_t* d_idx, int64_t k, const double* d_coef, int64_t m, double* d_out,
               cudaStream_t s) {
    if (geno_is_dense(g)) { dense_x_support(g, d_idx, k, d_coef, m, d_out, s); return; }
    // m right-hand sides in groups of <= 4 (coef is k x m column-major, out is n x m column-major)
    for (int64_t t0 = 0; t0 < m;) {
        int64_t mm = m - t0;
        const double* cf = d_coef + t0 * k;
        double* o = d_out + t0 * g->n;
        if (mm >= 4) { launch_x_support<4>(g, d_idx, k, cf, o, s); t0 += 4; }
        else if (mm == 3) { launch_x_support<3>(g, d_idx, k, cf, o, s); t0 += 3; }
        else if (mm == 2) { launch_x_support<2>(g, d_idx, k, cf, o, s); t0 += 2; }
        else { launch_x_support<1>(g, d_idx, k, cf, o, s); t0 += 1; }
    }
}

// Exact column dots. out[c + t*ncols] = sinv_j * (A + mu_j * (impute ? Mm : -vbar_t * nmiss_j)),
//   A = sum_{obs i} dos_ij (v_it - vbar_t), Mm = sum_{missing i} (v_it - vbar_t), j = cols[c].
// grid = (ncols, nsplit): each CTA reduces a contiguous byte range of one column with a fixed tree, a second tiny
// kernel adds the splits in order (deterministic, no atomics).
constexpr int XG_MAX_SPLIT = 64;


template <int M>
__global__ void __launch_bounds__(256)
k_xt_gather(GenoView gv, const int64_t* __restrict__ cols, int64_t n_a, const int64_t* __restrict__ cols_b,
            int64_t split_bytes, const double* __restrict__ v,
            const double* __restrict__ vbar, double* __restrict__ part /*[ncols][nsplit][2M]*/) {
    __shared__ double sh[32];
    const int64_t nbytes = gv.nbytes, n = gv.n;
    const int64_t c = blockIdx.x, sp = blockIdx.y;
    const int64_t j = c < n_a ? cols[c] : cols_b[c - n_a];      // two column lists, one launch (candidates | support)
    if (j < 0) return;                       // unused slot / column owned by another shard (block-uniform exit)
    const int64_t b0 = sp * split_bytes;
    const int64_t b1 = (b0 + split_bytes < nbytes) ? b0 + split_bytes : nbytes;
    double a[M], mm[M], vb[M];
#pragma unroll
    for (int t = 0; t < M; ++t) { a[t] = 0.0; mm[t] = 0.0; vb[t] = vbar[t]; }
    for (int64_t b = b0 + threadIdx.x; b < b1; b += blockDim.x) {
        uint32_t byte = *gv_ptr(gv, j, b);
        if (byte == 0) continue;
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            uint32_t code = (byte >> (2 * s)) & 3u;
            int64_t i = 4 * b + s;
            if (code != 0 && i < n) {
#pragma unroll
                for (int t = 0; t < M; ++t) {
                    double u = __dsub_rn(v[i + (int64_t)t * n], vb[t]);
                    if (code == 1) mm[t] = __dadd_rn(mm[t], u);
                    else a[t] = __dadd_rn(a[t], (code == 3) ? __dadd_rn(u, u) : u);
                }
            }
        }
    }
    double* o = part + (c * gridDim.y + sp) * (2 * M);
#pragma unroll
    for (int t = 0; t < M; ++t) {
        double at = block_sum(a[t], sh);
        double mt = block_sum(mm[t], sh);
        if (threadIdx.x == 0) { o[2 * t] = at; o[2 * t + 1] = mt; }
    }
}

template <int M>
__global__ void k_xt_gather_fin(GenoView gv, const int64_t* __restrict__ cols, int64_t n_a,
                                const int64_t* __restrict__ cols_b, int64_t ncols, int nsplit,
                                const double* __restrict__ vbar, const double* __restrict__ part,
                                double* __restrict__ out) {
    int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (e >= ncols * M) return;
    int64_t c = e / M;
    int t = (int)(e % M);
    const int64_t jc = c < n_a ? cols[c] : cols_b[c - n_a];
    if (jc < 0) { out[c + (int64_t)t * ncols] = 0.0; return; }
    double at = 0.0, mt = 0.0;
    for (int sp = 0; sp < nsplit; ++sp) {
        const double* o = part + (c * nsplit + sp) * (2 * M);
        at = __dadd_rn(at, o[2 * t]);
        mt = __dadd_rn(mt, o[2 * t + 1]);
    }
    int64_t j = jc;
    double corr = gv.impute ? mt : __dmul_rn(-vbar[t], (double)gv.nmiss[j]);
    out[c + (int64_t)t * ncols] = __dmul_rn(gv.sinv[j], __dadd_rn(at, __dmul_rn(gv.mu[j], corr)));
}

// Single right-hand side (every univariate fit): nibble tables.  A CTA owns one 512-sample chunk (one packed word per lane
// of a column) and builds, from the centred vector, T[k][nib][l] = dos(nib & 3) u[16 l + 2 k] + dos(nib >> 2) u[16 l + 2 k + 1]
// (k-th pair of samples of word l; code 01 = missing counts 0 here) -- 8 x 16 x 32 doubles = 32 KB, lane l reads bank pair l
// whatever the data.  Its 8 warps then walk the column list: per column and chunk a lane needs one 32-bit load, 8 table
// lookups and 8 FP64 adds for 16 genotypes, against ~13 instructions per genotype for a decode-and-select loop (the
// per-column kernel above also re-reads the vector for every column: 8 n bytes each from L2).  Measured at n = 500k,
// ~300 columns: 122 us -> see profiles/r2_gather_nibble.txt.  The sum over a column's MISSING samples that imputation
// needs comes from the handle's CSR list in the finalisation kernel, like in the sweep epilogue.
// One kernel for every list length, paired or solo fit, any number of shards: a column's value never depends on them.
constexpr int XN_CHUNK = 512;
__global__ void __launch_bounds__(256)
k_xt_gather_nib(GenoView gv, const int64_t* __restrict__ cols, int64_t n_a, const int64_t* __restrict__ cols_b,
                int64_t ncols, const double* __restrict__ v, const double* __restrict__ vbar,
                double* __restrict__ part /*[ncols][nchunks]*/) {
    __shared__ double T[8][16][32];                                 // 32 KB
    const int64_t n = gv.n;
    const int64_t chunk = blockIdx.x, nchunks = gridDim.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    {
        const double vb = vbar[0];
        const int64_t i0 = chunk * XN_CHUNK + 16 * lane + 2 * warp;             // thread (k = warp, l = lane) builds 16 rows
        const double u0 = (i0 < n) ? __dsub_rn(v[i0], vb) : 0.0;
        const double u1 = (i0 + 1 < n) ? __dsub_rn(v[i0 + 1], vb) : 0.0;
        const double d0[4] = {0.0, 0.0, u0, __dadd_rn(u0, u0)};
        const double d1[4] = {0.0, 0.0, u1, __dadd_rn(u1, u1)};
#pragma unroll
        for (int nib = 0; nib < 16; ++nib) T[warp][nib][lane] = __dadd_rn(d0[nib & 3], d1[nib >> 2]);
    }
    __syncthreads();
    const int64_t w = chunk * (XN_CHUNK / 16) + lane;               // this lane's packed word of a column
    const bool in_col = w < ((gv.nbytes + 3) >> 2);                 // bytes past nbytes inside a word are zero padding
    for (int64_t c = (int64_t)blockIdx.y * 8 + warp; c < ncols; c += (int64_t)gridDim.y * 8) {
        const int64_t j = c < n_a ? cols[c] : cols_b[c - n_a];
        if (j < 0) continue;                                        // unused slot / column of another shard
        const uint32_t x = in_col ? *reinterpret_cast<const uint32_t*>(gv_ptr(gv, j, 4 * w)) : 0u;
        double a = 0.0;
#pragma unroll
        for (int k = 0; k < 8; ++k) a = __dadd_rn(a, T[k][(x >> (4 * k)) & 15u][lane]);
        a = warp_sum(a);
        if (lane == 0) part[c * nchunks + chunk] = a;
    }
}

// one warp per column: lane l adds chunks l, l + 32, ... in order and its share of the column's missing samples (CSR),
// the lanes are combined by a fixed butterfly
__global__ void __launch_bounds__(128)
k_xt_gather_fin_nib(GenoView gv, const int64_t* __restrict__ miss_ptr, const int32_t* __restrict__ miss_idx,
                    const int64_t* __restrict__ cols, int64_t n_a, const int64_t* __restrict__ cols_b, int64_t ncols,
                    int nchunks, const double* __restrict__ v, const double* __restrict__ vbar,
                    const double* __restrict__ part, double* __restrict__ out) {
    const int64_t c = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (c >= ncols) return;
    const int64_t jc = c < n_a ? cols[c] : cols_b[c - n_a];
    if (jc < 0) { if (lane == 0) out[c] = 0.0; return; }
    double at = 0.0, mt = 0.0;
    for (int sp = lane; sp < nchunks; sp += 32) at = __dadd_rn(at, part[c * nchunks + sp]);
    const double vb = vbar[0];
    if (gv.impute)
        for (int64_t e = miss_ptr[jc] + lane; e < miss_ptr[jc + 1]; e += 32) mt = __dadd_rn(mt, __dsub_rn(v[miss_idx[e]], vb));
    at = warp_sum(at); mt = warp_sum(mt);
    if (lane == 0) {
        const double corr = gv.impute ? mt : __dmul_rn(-vb, (double)gv.nmiss[jc]);
        out[c] = __dmul_rn(gv.sinv[jc], __dadd_rn(at, __dmul_rn(gv.mu[jc], corr)));
    }
}

// split partial sums of the gather, one buffer per stream (a fit owns its stream; fits of several host threads and
// devices run concurrently, and the threads of a multi-device call are short-lived, so neither a global nor a
// thread-local buffer will do).  Buffers live until the process ends.
static DBuf<double>& gather_scratch(cudaStream_t s) {
    static std::mutex mu;
    static std::unordered_map<cudaStream_t, std::unique_ptr<DBuf<double>>> pool;
    std::lock_guard<std::mutex> lk(mu);
    auto& slot = pool[s];
    if (!slot) slot.reset(new DBuf<double>());
    return *slot;
}

template <int M>
static void launch_xt_gather(const ihtb_geno* g, const int64_t* d_cols, int64_t n_a, const int64_t* d_cols_b,
                             int64_t ncols, const double* d_v, const double* d_vbar, double* d_out, cudaStream_t s,
                             bool blocked) {
    DBuf<double>& sc = gather_scratch(s);
    (void)blocked;
    if (M == 1) {
        const int nchunks = (int)ceil_div(g->n, XN_CHUNK);
        const size_t need_b = (size_t)ncols * nchunks;
        if (sc.n < need_b) {
            IHTB_CUDA(cudaStreamSynchronize(s));
            sc.alloc(need_b < 65536 ? 65536 : need_b);
        }
        int groups = (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div(ncols, 8), (8 * g->sm_count) / nchunks + 1));
        IHTB_LAUNCH(k_xt_gather_nib, dim3((unsigned)nchunks, (unsigned)groups), 256, 0, s, geno_view(g), d_cols, n_a,
                    d_cols_b, ncols, d_v, d_vbar, sc.p);
        IHTB_LAUNCH(k_xt_gather_fin_nib, (unsigned)ceil_div(ncols * 32, 128), 128, 0, s, geno_view(g), g->miss_ptr.p,
                    g->miss_idx.p, d_cols, n_a, d_cols_b, ncols, nchunks, d_v, d_vbar, sc.p, d_out);
        return;
    }
    int64_t split_bytes = ceil_div(ceil_div(g->nbytes, XG_MAX_SPLIT), 256) * 256;
    if (split_bytes < 1024) split_bytes = 1024;
    int nsplit = (int)ceil_div(g->nbytes, split_bytes);
    size_t need = (size_t)ncols * nsplit * 2 * M;
    if (sc.n < need) {
        IHTB_CUDA(cudaStreamSynchronize(s));
        sc.alloc(need < 65536 ? 65536 : need);
    }
    dim3 grid((unsigned)ncols, (unsigned)nsplit);
    IHTB_LAUNCH((k_xt_gather<M>), grid, 256, 0, s, geno_view(g), d_cols, n_a, d_cols_b, split_bytes, d_v, d_vbar, sc.p);
    IHTB_LAUNCH((k_xt_gather_fin<M>), (unsigned)ceil_div(ncols * M, 128), 128, 0, s, geno_view(g), d_cols, n_a, d_cols_b,
                ncols, nsplit, d_vbar, sc.p, d_out);
}

// two column lists in one launch: out[0 .. n_a) from d_cols_a, out[n_a .. n_a + n_b) from d_cols_b (either may be empty)
void xt_gather2(const ihtb_geno* g, const int64_t* d_cols_a, int64_t n_a, const int64_t* d_cols_b, int64_t n_b,
                const double* d_v, int64_t m, const double* d_vbar, double* d_out, cudaStream_t s, bool blocked) {
    const int64_t ncols = n_a + n_b;
    if (ncols == 0) return;
    if (geno_is_dense(g)) { dense_xt_gather2(g, d_cols_a, n_a, d_cols_b, n_b, d_v, m, d_out, s); return; }   // plain dots
    for (int64_t t0 = 0; t0 < m;) {
        int64_t mm = m - t0;
        const double* vv = d_v + t0 * g->n;
        const double* vb = d_vbar + t0;
        double* o = d_out + t0 * ncols;
        if (mm >= 4) { launch_xt_gather<4>(g, d_cols_a, n_a, d_cols_b, ncols, vv, vb, o, s, blocked); t0 += 4; }
        else if (mm == 3) { launch_xt_gather<3>(g, d_cols_a, n_a, d_cols_b, ncols, vv, vb, o, s, blocked); t0 += 3; }
        else if (mm == 2) { launch_xt_gather<2>(g, d_cols_a, n_a, d_cols_b, ncols, vv, vb, o, s, blocked); t0 += 2; }
        else { launch_xt_gather<1>(g, d_cols_a, n_a, d_cols_b, ncols, vv, vb, o, s, blocked); t0 += 1; }
    }
}

void xt_gather(const ihtb_geno* g, const int64_t* d_cols, int64_t ncols, const double* d_v, int64_t m,
               const double* d_vbar, double* d_out, cudaStream_t s) {
    xt_gather2(g, d_cols, ncols, nullptr, 0, d_v, m, d_vbar, d_out, s, false);
}

}  // namespace ihtb

using namespace ihtb;

// Diagnostic / bench entry: exact column dots X[:, cols]' v for ncols columns (j_t = (t * 7919) mod p) through the
// nibble-table kernel (what every univariate fit uses), timed, and checked against the per-column decode kernel
// (run with two identical right-hand sides, which takes the other code path).  v is a fixed pseudo-random vector.
__global__ void k_gb_fill(double* v, int64_t n) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) {
        uint64_t h = (uint64_t)i * 0x9E3779B97F4A7C15ull + 12345ull;
        h ^= h >> 31; h *= 0xBF58476D1CE4E5B9ull; h ^= h >> 29;
        v[i] = (double)(h >> 11) * (1.0 / 9007199254740992.0) - 0.4;
        v[i + n] = v[i];
    }
}
extern "C" int32_t ihtb_gather_bench(const ihtb_geno* g, int64_t ncols, int32_t reps, double* ms_per_call,
                                     double* max_rel_diff) {
    return guard([&] {
        IHTB_CHECK(g && ncols >= 1 && reps >= 1, IHTB_EINVAL, "bad argument");
        IHTB_CHECK(!geno_is_dense(g), IHTB_EUNSUPPORTED, "the gather bench times the PLINK re-scoring kernels");
        geno_require_ready(g);
        IHTB_CUDA(cudaSetDevice(g->device));
        cudaStream_t s;
        IHTB_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
        std::vector<int64_t> hc((size_t)ncols);
        for (int64_t t = 0; t < ncols; ++t) hc[(size_t)t] = (t * 7919) % g->p;
        DBuf<int64_t> d_cols((size_t)ncols);
        DBuf<double> d_v((size_t)(2 * g->n)), d_mean(2), d_a((size_t)ncols), d_b((size_t)(2 * ncols));
        IHTB_CUDA(cudaMemcpyAsync(d_cols.p, hc.data(), (size_t)ncols * sizeof(int64_t), cudaMemcpyHostToDevice, s));
        IHTB_LAUNCH(k_gb_fill, (unsigned)ceil_div(g->n, 256), 256, 0, s, d_v.p, g->n);
        const double mean[2] = {0.1, 0.1};                       // any centring value: both kernels subtract the same one
        IHTB_CUDA(cudaMemcpyAsync(d_mean.p, mean, sizeof(mean), cudaMemcpyHostToDevice, s));
        xt_gather2(g, d_cols.p, ncols, nullptr, 0, d_v.p, 1, d_mean.p, d_a.p, s);            // warm-up (scratch)
        cudaEvent_t e0, e1;
        IHTB_CUDA(cudaEventCreate(&e0)); IHTB_CUDA(cudaEventCreate(&e1));
        IHTB_CUDA(cudaEventRecord(e0, s));
        for (int i = 0; i < reps; ++i) xt_gather2(g, d_cols.p, ncols, nullptr, 0, d_v.p, 1, d_mean.p, d_a.p, s);
        IHTB_CUDA(cudaEventRecord(e1, s));
        xt_gather2(g, d_cols.p, ncols, nullptr, 0, d_v.p, 2, d_mean.p, d_b.p, s);            // per-column decode kernel
        std::vector<double> ha((size_t)ncols), hb((size_t)(2 * ncols));
        IHTB_CUDA(cudaMemcpyAsync(ha.data(), d_a.p, ha.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
        IHTB_CUDA(cudaMemcpyAsync(hb.data(), d_b.p, hb.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
        IHTB_CUDA(cudaStreamSynchronize(s));
        float ms = 0.f;
        IHTB_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        if (ms_per_call) *ms_per_call = ms / reps;
        double worst = 0.0, scale = 0.0;
        for (int64_t t = 0; t < ncols; ++t) scale = std::max(scale, std::fabs(hb[(size_t)t]));
        for (int64_t t = 0; t < ncols; ++t) worst = std::max(worst, std::fabs(ha[(size_t)t] - hb[(size_t)t]));
        if (max_rel_diff) *max_rel_diff = scale > 0 ? worst / scale : worst;
        cudaEventDestroy(e0); cudaEventDestroy(e1);
        cudaStreamDestroy(s);
    });
}

extern "C" int32_t ihtb_x_support(const ihtb_geno* g, const int64_t* idx, int64_t k, const double* coef, int64_t m,
                                  double* out) {
    return guard([&] {
        IHTB_CHECK(g && out && m >= 1 && k >= 0, IHTB_EINVAL, "bad argument");
        geno_require_ready(g);
        IHTB_CHECK(k == 0 || (idx && coef), IHTB_EINVAL, "NULL idx/coef");
        IHTB_CUDA(cudaSetDevice(g->device));
        for (int64_t c = 0; c < k; ++c)
            IHTB_CHECK(idx[c] >= 0 && idx[c] < g->p, IHTB_EDIM, "support index out of range");
        DBuf<double> d_out((size_t)(g->n * m));
        if (k == 0) {
            d_out.zero(0);
        } else {
            DBuf<int64_t> d_idx((size_t)k);
            DBuf<double> d_coef((size_t)(k * m));
            IHTB_CUDA(cudaMemcpy(d_idx.p, idx, k * sizeof(int64_t), cudaMemcpyHostToDevice));
            IHTB_CUDA(cudaMemcpy(d_coef.p, coef, k * m * sizeof(double), cudaMemcpyHostToDevice));
            x_support(g, d_idx.p, k, d_coef.p, m, d_out.p, 0);
        }
        IHTB_CUDA(cudaMemcpy(out, d_out.p, g->n * m * sizeof(double), cudaMemcpyDeviceToHost));
    });
}
