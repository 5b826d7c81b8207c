// Genotype handle: device-resident 2-bit PLINK matrix + per-SNP statistics.
// Replaces SnpLinAlg{Float64}(s; model=ADDITIVE_MODEL, center, scale, impute) (constructed at reference
// src/wrapper.jl:68-69,318-319; SnpArrays.jl itself is an external dependency, semantics in SURVEY.md App. A.1).
#include "common.cuh"
#include "synth.cuh"
#include <mutex>
#include <thread>
#include <stdlib.h>
#include <string.h>

extern "C" void ihtb_internal_fit_cache_clear(int device);

namespace ihtb {

static thread_local std::string t_last_error;
void set_last_error(const std::string& m) { t_last_error = m; }
const std::string& last_error() { return t_last_error; }
LaunchCounter& launch_counter() {
    static LaunchCounter c;
    return c;
}
bool smem_attr_needed(const void* kernel, int device) {
    static std::mutex mu;
    static std::vector<std::pair<const void*, int>> done;
    std::lock_guard<std::mutex> lk(mu);
    for (const auto& e : done)
        if (e.first == kernel && e.second == device) return false;
    done.push_back({kernel, device});
    return true;
}
bool debug_sync() {
    static int v = -1;
    if (v < 0) { const char* e = getenv("IHTB_DEBUG_SYNC"); v = (e && *e == '1') ? 1 : 0; }
    return v == 1;
}

// ---------------------------------------------------------------------------------------------
// Kernels
// ---------------------------------------------------------------------------------------------

// zero the unused high bits of the last data byte of every column (n % 4 != 0)
__global__ void k_mask_tail(GenoView g, int n_rem) {
    int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (j >= g.p) return;
    uint8_t mask = (uint8_t)((1u << (2 * n_rem)) - 1u);
    *const_cast<uint8_t*>(gv_ptr(g, j, g.nbytes - 1)) &= mask;
}

// repack a column-major staging block (columns [j0, j0+ncols), `nbytes` bytes each, pitch `pitch`) into the handle's
// layout, 16 bytes per thread; the tail of the last 16-byte vector of a column is zero-filled
__global__ void k_repack(const uint8_t* __restrict__ staging, int64_t pitch, int64_t j0, int64_t ncols, GenoView g) {
    int64_t vec_per_col = (g.nbytes + 15) >> 4;
    int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= ncols * vec_per_col) return;
    int64_t c = t / vec_per_col, v = t % vec_per_col;
    const uint8_t* src = staging + c * pitch + 16 * v;
    uint8_t tmp[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) tmp[k] = (16 * v + k < g.nbytes) ? src[k] : (uint8_t)0;
    uint32_t q[4];
    memcpy(q, tmp, 16);
#pragma unroll
    for (int k = 0; k < 4; ++k)      // words are the contiguous unit of every layout (gv_ptr)
        *reinterpret_cast<uint32_t*>(const_cast<uint8_t*>(gv_ptr(g, j0 + c, 16 * v + 4 * k))) = q[k];
}

// inverse of k_repack for export: out[c][b] = byte b of column j0 + c
__global__ void k_export(GenoView g, int64_t j0, int64_t ncols, uint8_t* __restrict__ out) {
    int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= ncols * g.nbytes) return;
    int64_t c = t / g.nbytes, b = t % g.nbytes;
    out[t] = *gv_ptr(g, j0 + c, b);
}

// one warp per column: counts of het (10), hom2 (11), missing (01) -> mu, sigma_inv
// mu_j = (n1 + 2 n2) / n_obs ; sigma_inv_j = 1/sqrt(mu_j (1 - mu_j/2)) or 1 (same statistic as the
// reference's standardize_genotypes!, src/wrapper.jl:409-416)
__global__ void k_col_stats(GenoView g, int scale, double* __restrict__ mu, double* __restrict__ sinv,
                            int32_t* __restrict__ nmiss, double* __restrict__ sgn) {
    int64_t j = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (j >= g.p) return;
    const int64_t n = g.n;
    int64_t nvec = g.stride >> 4;
    int c1 = 0, c2 = 0, cm = 0;
    for (int64_t v = lane; v < nvec; v += 32) {
        uint32_t w[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) w[t] = *reinterpret_cast<const uint32_t*>(gv_ptr(g, j, 16 * v + 4 * t));
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            uint32_t lo = w[t] & 0x55555555u, hi = (w[t] >> 1) & 0x55555555u;
            cm += __popc(lo & ~hi);
            c1 += __popc(hi & ~lo);
            c2 += __popc(hi & lo);
        }
    }
    c1 = warp_sum(c1); c2 = warp_sum(c2); cm = warp_sum(cm);
    if (lane == 0) {
        double nobs = (double)(n - cm);
        double m = (double)((int64_t)c1 + 2 * (int64_t)c2) / nobs;
        double s = sqrt(__dmul_rn(m, __dsub_rn(1.0, m / 2.0)));
        mu[j] = m;
        const double si = (scale && s > 0.0) ? 1.0 / s : 1.0;
        sinv[j] = si;
        nmiss[j] = cm;
        const double g2 = sqrt((double)((int64_t)c1 + 4 * (int64_t)c2));      // sqrt(sum of squared dosages)
        sgn[j] = si * (g2 > 1.0 ? g2 : 1.0);
    }
}

// one warp per column: how many samples carry each 2-bit code (SnpArrays `counts(s, dims=1)`: rows 00, 01 = missing, 10, 11)
__global__ void k_col_counts(GenoView g, int64_t* __restrict__ out /*[4][p] column-major 4 x p*/) {
    int64_t j = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (j >= g.p) return;
    int64_t nvec = g.stride >> 4;
    int c1 = 0, c2 = 0, cm = 0;
    for (int64_t v = lane; v < nvec; v += 32) {
        uint32_t w[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) w[t] = *reinterpret_cast<const uint32_t*>(gv_ptr(g, j, 16 * v + 4 * t));
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            uint32_t lo = w[t] & 0x55555555u, hi = (w[t] >> 1) & 0x55555555u;
            cm += __popc(lo & ~hi);
            c1 += __popc(hi & ~lo);
            c2 += __popc(hi & lo);
        }
    }
    c1 = warp_sum(c1); c2 = warp_sum(c2); cm = warp_sum(cm);
    if (lane == 0) {
        out[4 * j + 0] = g.n - c1 - c2 - cm;      // padding beyond n is zero-filled = code 00, hence n - others
        out[4 * j + 1] = cm;
        out[4 * j + 2] = c1;
        out[4 * j + 3] = c2;
    }
}

// CSR fill of missing sample indices: one warp per column, ordered by sample index
__global__ void k_fill_missing(GenoView g, const int64_t* __restrict__ ptr, int32_t* __restrict__ idx) {
    int64_t j = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (j >= g.p) return;
    int64_t base = ptr[j];
    if (ptr[j + 1] == base) return;
    const int64_t nbytes = g.nbytes;
    int64_t off = 0;
    for (int64_t b0 = 0; b0 < nbytes; b0 += 32) {
        int64_t b = b0 + lane;
        uint32_t byte = (b < nbytes) ? *gv_ptr(g, j, b) : 0u;
        uint32_t lo = byte & 0x55u, hi = (byte >> 1) & 0x55u;
        uint32_t mm = lo & ~hi;  // bit 2t set if sample t of this byte is missing
        int cnt = __popc(mm);
        // exclusive prefix over lanes
        int pre = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int t = __shfl_up_sync(0xffffffffu, pre, o);
            if (lane >= o) pre += t;
        }
        int total = __shfl_sync(0xffffffffu, pre, 31);
        pre -= cnt;
        int w = 0;
#pragma unroll
        for (int t = 0; t < 4; ++t)
            if (mm & (1u << (2 * t))) idx[base + off + pre + (w++)] = (int32_t)(4 * b + t);
        off += total;
    }
}

// bit-exact getindex: x_ij = ((missing ? mu_j : g_ij) - mu_j) * sigma_inv_j
__global__ void k_decode(GenoView gv, int center, int64_t i0, int64_t i1, int64_t j0, int64_t j1,
                         double* __restrict__ out) {
    int64_t ni = i1 - i0;
    int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= ni * (j1 - j0)) return;
    int64_t j = j0 + t / ni, i = i0 + t % ni;
    uint32_t code = (*gv_ptr(gv, j, i >> 2) >> (2 * (i & 3))) & 3u;
    double m = gv.mu[j];
    double g = (code == 2) ? 1.0 : (code == 3) ? 2.0 : (code == 1) ? (gv.impute ? m : 0.0) : 0.0;
    if (center) g = __dsub_rn(g, m);
    out[t] = __dmul_rn(g, gv.sinv[j]);
}

// synthetic generator: one thread per 32-bit word (16 samples) of a column
__global__ void k_synth(GenoView g, int64_t j0, uint64_t seed, uint32_t miss_thr) {
    const int64_t n = g.n;
    int64_t words = g.stride >> 2;
    int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= g.p * words) return;
    int64_t j = t / words, w = t % words;
    uint64_t key = synth_col_key(seed, (uint64_t)(j0 + j));
    uint64_t thr = synth_maf_threshold(key);
    uint32_t out = 0;
#pragma unroll
    for (int s = 0; s < 16; ++s) {
        int64_t i = 16 * w + s;
        if (i < n) out |= synth_code(key, thr, miss_thr, (uint64_t)i) << (2 * s);
    }
    *reinterpret_cast<uint32_t*>(const_cast<uint8_t*>(gv_ptr(g, j, 4 * w))) = out;
}

// Ternary copy of the quad-interleaved tiles (common.cuh ihtb_geno::tern): thread = one 32-bit word of the copy =
// 20 samples of one column = 5 source bytes.  idx = ((slab * nquads + quad) * 32 + w) * 4 + cj, so stores are coalesced.
// Component cj of the 16 bytes at word position w holds column 4 quad + (cj ^ (w & 3)): lane w of a sweep warp then finds
// its accumulator slots already arranged for a select-free butterfly (sweep_lut.cu).  Only the sweeps read this copy.
__global__ void k_make_tern(GenoView g, int64_t p4, int64_t tern_slabs, uint32_t* __restrict__ out) {
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t total = tern_slabs * p4 * 32;
    if (idx >= total) return;
    const int cj = (int)(idx & 3), w = (int)((idx >> 2) & 31);
    const int64_t sq = idx >> 7, nquads = p4 >> 2;
    const int64_t slab = sq / nquads, j = (sq % nquads) * 4 + (cj ^ (w & 3));
    uint32_t word = 0;
    if (j < g.p) {
        const int64_t b0 = slab * 160 + 5 * w;                  // first of the 5 source bytes (20 samples)
        uint32_t code[20];
#pragma unroll
        for (int t = 0; t < 5; ++t) {
            const int64_t b = b0 + t;
            const uint32_t byte = b < g.stride ? *gv_ptr(g, j, b) : 0u;      // bytes past nbytes are zero padding
#pragma unroll
            for (int s = 0; s < 4; ++s) code[4 * t + s] = (byte >> (2 * s)) & 3u;
        }
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            uint32_t v = 0;
#pragma unroll
            for (int d = 4; d >= 0; --d) {
                const uint32_t c = code[5 * t + d];
                v = 3u * v + ((c >> 1) * (1u + (c & 1u)));       // 00 -> 0, 01 (missing) -> 0, 10 -> 1, 11 -> 2
            }
            word |= v << (8 * t);
        }
    }
    out[idx] = word;
}

// ---------------------------------------------------------------------------------------------
// Host side
// ---------------------------------------------------------------------------------------------
// IHTB_TERN=0 never builds the ternary copy, =1 always; default: when it takes at most half of the memory still free
// (a 125 GB matrix on one GPU keeps the 2-bit sweep; its column shards on 8 GPUs get the copy)
static void build_tern(ihtb_geno* g, cudaStream_t s) {
    g->tern.release();
    g->tern_slabs = 0;
    if (!g->quad) return;
    const char* e = getenv("IHTB_TERN");
    if (e && *e == '0') return;
    const int64_t slabs = ceil_div(g->n, 640);
    const size_t bytes = (size_t)slabs * (size_t)g->p4 * 128;
    if (!(e && *e == '1')) {
        size_t free_b = 0, total_b = 0;
        IHTB_CUDA(cudaMemGetInfo(&free_b, &total_b));
        if (bytes > free_b / 2) return;
    }
    g->tern.alloc(bytes);
    g->tern_slabs = slabs;
    const int64_t words = slabs * g->p4 * 32;
    IHTB_LAUNCH(k_make_tern, (unsigned)ceil_div(words, 256), 256, 0, s, geno_view(g), g->p4, slabs,
                reinterpret_cast<uint32_t*>(g->tern.p));
}

static void finish_handle(ihtb_geno* g) {
    cudaStream_t s = 0;
    g->mu.alloc(g->p); g->sinv.alloc(g->p); g->nmiss.alloc(g->p); g->sgn.alloc(g->p);
    int64_t threads = g->p * 32;
    IHTB_LAUNCH(k_col_stats, (unsigned)ceil_div(threads, 256), 256, 0, s, geno_view(g), g->scale, g->mu.p, g->sinv.p,
                g->nmiss.p, g->sgn.p);
    g->miss_ptr.alloc(g->p + 1);
    int64_t total = 0;
    {   // exclusive scan of the per-column missing counts (host: once per handle, p <= a few million)
        std::vector<int32_t> hn((size_t)g->p);
        std::vector<int64_t> hp((size_t)g->p + 1);
        IHTB_CUDA(cudaMemcpy(hn.data(), g->nmiss.p, g->p * sizeof(int32_t), cudaMemcpyDeviceToHost));
        for (int64_t j = 0; j < g->p; ++j) { hp[j] = total; total += hn[j]; }
        hp[g->p] = total;
        IHTB_CUDA(cudaMemcpy(g->miss_ptr.p, hp.data(), (g->p + 1) * sizeof(int64_t), cudaMemcpyHostToDevice));
    }
    g->total_missing = total;
    if (total > 0) {
        g->miss_idx.alloc(total);
        IHTB_LAUNCH(k_fill_missing, (unsigned)ceil_div(threads, 256), 256, 0, s, geno_view(g), g->miss_ptr.p,
                    g->miss_idx.p);
    }
    build_tern(g, s);
    IHTB_CUDA(cudaStreamSynchronize(s));
}

static ihtb_geno* new_handle(int64_t n, int64_t p, int center, int scale, int impute) {
    IHTB_CHECK(n > 0 && p > 0, IHTB_EDIM, "genotype matrix must have n > 0 and p > 0");
    IHTB_CHECK(n < (int64_t(1) << 31), IHTB_EDIM, "n must be < 2^31");
    IHTB_CHECK(center == 1, IHTB_EUNSUPPORTED,
               "x is not centered! Please construct SnpLinAlg{Float64}(::SnpArray, center=true, scale=true)");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        throw Error(IHTB_ECUDA, "no CUDA device available (libihtb200 has no CPU fallback)");
    ihtb_geno* g = new ihtb_geno();
    IHTB_CUDA(cudaGetDevice(&g->device));
    IHTB_CUDA(cudaDeviceGetAttribute(&g->sm_count, cudaDevAttrMultiProcessorCount, g->device));
    g->n = n; g->p = p;
    g->nbytes = (n + 3) / 4;
    g->stride = ceil_div(g->nbytes, 128) * 128;
    // HBM layout (common.cuh): quad-interleaved slab-major tiles by default; IHTB_LAYOUT=tiled keeps plain 128-byte
    // tiles (the round-1 TMA sweep), IHTB_LAYOUT=colmajor PLINK's column-major order (padded stride, debug only)
    const char* lay = getenv("IHTB_LAYOUT");
    g->p4 = (p + 3) / 4 * 4;
    if (lay && std::string(lay) == "colmajor") { g->cs_j = g->stride; g->cs_s = 128; g->p4 = p; }
    else if (lay && std::string(lay) == "tiled") { g->cs_j = 128; g->cs_s = g->p * 128; g->p4 = p; }
    else { g->quad = 1; g->cs_j = 128; g->cs_s = g->p4 * 128; }
    g->center = center; g->scale = scale; g->impute = impute;
    try {
        g->bed.alloc((size_t)(g->p4 * g->stride));
        if (g->p4 != g->p) IHTB_CUDA(cudaMemset(g->bed.p, 0, (size_t)(g->p4 * g->stride)));   // padding columns
    } catch (...) {
        delete g;
        throw;
    }
    return g;
}

}  // namespace ihtb

using namespace ihtb;

extern "C" {

int32_t ihtb_version(void) { return 100; }

int32_t ihtb_last_error(char* buf, int64_t cap) {
    if (!buf || cap <= 0) return IHTB_EINVAL;
    const std::string& m = ihtb::last_error();
    int64_t k = (int64_t)m.size() < cap - 1 ? (int64_t)m.size() : cap - 1;
    memcpy(buf, m.data(), (size_t)k);
    buf[k] = 0;
    return IHTB_OK;
}

int32_t ihtb_device_count(int32_t* count) {
    return guard([&] {
        IHTB_CHECK(count, IHTB_EINVAL, "count is NULL");
        int n = 0;
        cudaError_t e = cudaGetDeviceCount(&n);
        *count = (e == cudaSuccess) ? n : 0;
        if (e != cudaSuccess) cudaGetLastError();
    });
}

int32_t ihtb_set_device(int32_t device) {
    return guard([&] { IHTB_CUDA(cudaSetDevice(device)); });
}

int32_t ihtb_launch_count(int64_t* count) {
    return guard([&] {
        IHTB_CHECK(count, IHTB_EINVAL, "count is NULL");
        *count = launch_counter();
    });
}

// Host -> HBM ingest of `ncols` PLINK columns starting at local column j_dst.  Two pinned buffers: while chunk i is
// copied to the device and repacked into the tiled layout on `st`, a pool of host threads gathers chunk i+1 from the
// caller's (typically mmapped, page-faulting) memory into the other buffer, so file I/O, PCIe and the repack overlap
// and the resident host footprint is bounded (2 x 64 MiB) whatever the file size (SURVEY.md 8f2).
static void upload_columns(ihtb_geno* g, const uint8_t* bed_cols, int64_t col_stride_bytes, int64_t j_dst, int64_t ncols) {
    const int64_t pitch = ceil_div(g->nbytes, 16) * 16;
    int64_t cols_per = (int64_t(64) << 20) / pitch;
    if (cols_per < 1) cols_per = 1;
    if (cols_per > ncols) cols_per = ncols;
    const int NB = 2;
    HBuf<uint8_t> hbuf[NB];
    DBuf<uint8_t> dbuf[NB];
    cudaEvent_t done[NB];
    cudaStream_t st;
    IHTB_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    for (int b = 0; b < NB; ++b) {
        hbuf[b].alloc((size_t)(cols_per * pitch));
        dbuf[b].alloc((size_t)(cols_per * pitch));
        IHTB_CUDA(cudaEventCreateWithFlags(&done[b], cudaEventDisableTiming));
    }
    unsigned nt = std::thread::hardware_concurrency();
    if (nt == 0) nt = 1;
    if (nt > 16) nt = 16;
    const GenoView gv = geno_view(g);
    const int64_t vec_per_col = (g->nbytes + 15) >> 4;
    const int64_t nbytes = g->nbytes;
    int b = 0;
    try {
        for (int64_t j = 0; j < ncols; j += cols_per, b ^= 1) {
            const int64_t h = (ncols - j < cols_per) ? ncols - j : cols_per;
            IHTB_CUDA(cudaEventSynchronize(done[b]));                 // buffer b is free again
            uint8_t* dst = hbuf[b].p;
            const uint8_t* src = bed_cols + j * col_stride_bytes;
            const unsigned use = (unsigned)std::min<int64_t>(nt, h);
            std::vector<std::thread> pool;
            for (unsigned t = 1; t < use; ++t)
                pool.emplace_back([=] {
                    for (int64_t c = h * t / use; c < h * (t + 1) / use; ++c)
                        memcpy(dst + c * pitch, src + c * col_stride_bytes, (size_t)nbytes);
                });
            for (int64_t c = 0; c < h / use; ++c) memcpy(dst + c * pitch, src + c * col_stride_bytes, (size_t)nbytes);
            for (auto& th : pool) th.join();
            IHTB_CUDA(cudaMemcpyAsync(dbuf[b].p, hbuf[b].p, (size_t)(h * pitch), cudaMemcpyHostToDevice, st));
            IHTB_LAUNCH(k_repack, (unsigned)ceil_div(h * vec_per_col, 256), 256, 0, st, dbuf[b].p, pitch, j_dst + j, h, gv);
            IHTB_CUDA(cudaEventRecord(done[b], st));
        }
        IHTB_CUDA(cudaStreamSynchronize(st));
    } catch (...) {
        cudaStreamSynchronize(st);
        for (int i = 0; i < NB; ++i) cudaEventDestroy(done[i]);
        cudaStreamDestroy(st);
        throw;
    }
    for (int i = 0; i < NB; ++i) cudaEventDestroy(done[i]);
    cudaStreamDestroy(st);
}

static void seal_handle(ihtb_geno* g) {
    if (g->n % 4) IHTB_LAUNCH(k_mask_tail, (unsigned)ceil_div(g->p, 256), 256, 0, 0, geno_view(g), (int)(g->n % 4));
    finish_handle(g);
    g->ready = true;
}

int32_t ihtb_geno_create(const uint8_t* bed_cols, int64_t n, int64_t p, int64_t col_stride_bytes, int32_t center,
                         int32_t scale, int32_t impute, ihtb_geno** out) {
    return guard([&] {
        IHTB_CHECK(bed_cols && out, IHTB_EINVAL, "NULL argument");
        IHTB_CHECK(col_stride_bytes >= (n + 3) / 4, IHTB_EDIM, "col_stride_bytes is smaller than ceil(n/4)");
        ihtb_geno* g = new_handle(n, p, center, scale, impute);
        try {
            IHTB_CUDA(cudaMemset(g->bed.p, 0, (size_t)(g->p4 * g->stride)));
            upload_columns(g, bed_cols, col_stride_bytes, 0, p);
            seal_handle(g);
        } catch (...) {
            delete g;
            throw;
        }
        *out = g;
    });
}

// ---- piecewise ingest: per-chromosome files, or sources that cannot be mapped as one array -----------------------
int32_t ihtb_geno_create_empty(int64_t n, int64_t p, int32_t center, int32_t scale, int32_t impute, ihtb_geno** out) {
    return guard([&] {
        IHTB_CHECK(out, IHTB_EINVAL, "NULL argument");
        ihtb_geno* g = new_handle(n, p, center, scale, impute);
        try {
            IHTB_CUDA(cudaMemset(g->bed.p, 0, (size_t)(g->p4 * g->stride)));
        } catch (...) {
            delete g;
            throw;
        }
        g->ready = false;
        *out = g;
    });
}

int32_t ihtb_geno_load_columns(ihtb_geno* g, const uint8_t* bed_cols, int64_t col_stride_bytes, int64_t j_first,
                               int64_t ncols) {
    return guard([&] {
        IHTB_CHECK(g && bed_cols, IHTB_EINVAL, "NULL argument");
        IHTB_CHECK(!geno_is_dense(g), IHTB_EINVAL, "a dense handle takes ihtb_geno_load_dense_columns");
        IHTB_CHECK(!g->ready, IHTB_EINVAL, "genotype handle is already finalized");
        IHTB_CHECK(col_stride_bytes >= g->nbytes, IHTB_EDIM, "col_stride_bytes is smaller than ceil(n/4)");
        IHTB_CHECK(j_first >= 0 && ncols >= 0 && j_first + ncols <= g->p, IHTB_EDIM, "column range outside the matrix");
        IHTB_CUDA(cudaSetDevice(g->device));
        if (ncols > 0) upload_columns(g, bed_cols, col_stride_bytes, j_first, ncols);
    });
}

int32_t ihtb_geno_finalize(ihtb_geno* g) {
    return guard([&] {
        IHTB_CHECK(g, IHTB_EINVAL, "NULL argument");
        IHTB_CHECK(!g->ready, IHTB_EINVAL, "genotype handle is already finalized");
        IHTB_CUDA(cudaSetDevice(g->device));
        if (geno_is_dense(g)) {
            dense_finalize(g);
            g->ready = true;
        } else {
            seal_handle(g);
        }
    });
}

int32_t ihtb_geno_create_synthetic(int64_t n, int64_t p_local, int64_t j0, uint64_t seed, double missing_rate,
                                   ihtb_geno** out) {
    return guard([&] {
        IHTB_CHECK(out, IHTB_EINVAL, "NULL argument");
        IHTB_CHECK(missing_rate >= 0.0 && missing_rate < 1.0, IHTB_EINVAL, "missing_rate must be in [0, 1)");
        ihtb_geno* g = new_handle(n, p_local, 1, 1, 1);
        try {
            g->j0 = j0;
            uint32_t miss_thr = synth_missing_threshold(missing_rate);
            int64_t words = g->stride >> 2;
            int64_t total = g->p * words;
            IHTB_LAUNCH(k_synth, (unsigned)ceil_div(total, 256), 256, 0, 0, geno_view(g), j0, seed, miss_thr);
            finish_handle(g);
            g->ready = true;
        } catch (...) {
            delete g;
            throw;
        }
        *out = g;
    });
}

// host twin of k_synth (multi-threaded); lets callers build host-resident .bed columns identical to the device ones
int32_t ihtb_synth_host(int64_t n, int64_t ncols, int64_t j0, uint64_t seed, double missing_rate, uint8_t* out) {
    return guard([&] {
        IHTB_CHECK(out && n > 0 && ncols >= 0, IHTB_EINVAL, "bad argument");
        const int64_t nbytes = (n + 3) / 4;
        const uint32_t miss_thr = synth_missing_threshold(missing_rate);
        unsigned nt = std::thread::hardware_concurrency();
        if (nt == 0) nt = 1;
        if ((int64_t)nt > ncols) nt = (unsigned)(ncols > 0 ? ncols : 1);
        std::vector<std::thread> pool;
        for (unsigned t = 0; t < nt; ++t) {
            pool.emplace_back([=] {
                for (int64_t c = ncols * t / nt; c < ncols * (t + 1) / nt; ++c) {
                    uint64_t key = synth_col_key(seed, (uint64_t)(j0 + c));
                    uint64_t thr = synth_maf_threshold(key);
                    uint8_t* col = out + c * nbytes;
                    for (int64_t b = 0; b < nbytes; ++b) {
                        uint32_t byte = 0;
                        for (int s = 0; s < 4; ++s) {
                            int64_t i = 4 * b + s;
                            if (i < n) byte |= synth_code(key, thr, miss_thr, (uint64_t)i) << (2 * s);
                        }
                        col[b] = (uint8_t)byte;
                    }
                }
            });
        }
        for (auto& th : pool) th.join();
    });
}

int32_t ihtb_geno_sweep_stream_bytes(const ihtb_geno* g, int64_t* bytes, int32_t* ternary) {
    return guard([&] {
        IHTB_CHECK(g, IHTB_EINVAL, "NULL genotype handle");
        geno_require_ready(g);
        if (geno_is_dense(g)) {
            if (bytes) *bytes = dense_stream_bytes(g);
            if (ternary) *ternary = 0;
            return;
        }
        const bool t = g->tern.p != nullptr;
        if (bytes) *bytes = (t ? g->tern_slabs : g->stride / 128) * g->p4 * 128;
        if (ternary) *ternary = t ? 1 : 0;
    });
}

int32_t ihtb_geno_set_offset(ihtb_geno* g, int64_t j0) {
    return guard([&] {
        IHTB_CHECK(g && j0 >= 0, IHTB_EINVAL, "bad argument");
        IHTB_CHECK(!geno_is_dense(g), IHTB_EUNSUPPORTED, "dense handles cannot be SNP shards");
        g->j0 = j0;
    });
}

int32_t ihtb_geno_dims(const ihtb_geno* g, int64_t* n, int64_t* p) {
    return guard([&] {
        IHTB_CHECK(g, IHTB_EINVAL, "NULL genotype handle");
        if (n) *n = g->n;
        if (p) *p = g->p;
    });
}

int32_t ihtb_geno_stats(const ihtb_geno* g, double* mu, double* sigma_inv, int64_t* n_missing) {
    return guard([&] {
        IHTB_CHECK(g, IHTB_EINVAL, "NULL genotype handle");
        geno_require_ready(g);
        IHTB_CUDA(cudaSetDevice(g->device));
        if (mu) IHTB_CUDA(cudaMemcpy(mu, g->mu.p, g->p * sizeof(double), cudaMemcpyDeviceToHost));
        if (sigma_inv) IHTB_CUDA(cudaMemcpy(sigma_inv, g->sinv.p, g->p * sizeof(double), cudaMemcpyDeviceToHost));
        if (n_missing) {
            std::vector<int32_t> tmp(g->p);
            IHTB_CUDA(cudaMemcpy(tmp.data(), g->nmiss.p, g->p * sizeof(int32_t), cudaMemcpyDeviceToHost));
            for (int64_t j = 0; j < g->p; ++j) n_missing[j] = tmp[j];
        }
    });
}

int32_t ihtb_geno_counts(const ihtb_geno* g, int64_t* counts) {
    return guard([&] {
        IHTB_CHECK(g && counts, IHTB_EINVAL, "NULL argument");
        IHTB_CHECK(!geno_is_dense(g), IHTB_EUNSUPPORTED, "genotype counts need a PLINK handle");
        geno_require_ready(g);
        IHTB_CUDA(cudaSetDevice(g->device));
        DBuf<int64_t> d((size_t)(4 * g->p));
        IHTB_LAUNCH(k_col_counts, (unsigned)ceil_div(g->p * 32, 256), 256, 0, 0, geno_view(g), d.p);
        IHTB_CUDA(cudaMemcpy(counts, d.p, (size_t)(4 * g->p) * sizeof(int64_t), cudaMemcpyDeviceToHost));
    });
}

int32_t ihtb_geno_maf(const ihtb_geno* g, double* maf) {
    return guard([&] {
        IHTB_CHECK(g && maf, IHTB_EINVAL, "NULL argument");
        IHTB_CHECK(!geno_is_dense(g), IHTB_EUNSUPPORTED, "maf needs a PLINK handle (SnpArray)");
        geno_require_ready(g);
        IHTB_CUDA(cudaSetDevice(g->device));
        IHTB_CUDA(cudaMemcpy(maf, g->mu.p, g->p * sizeof(double), cudaMemcpyDeviceToHost));
        for (int64_t j = 0; j < g->p; ++j) {          // (n1 + 2 n2) / (2 n_obs), folded to the minor allele
            double f = maf[j] / 2.0;
            maf[j] = f > 0.5 ? 1.0 - f : f;
        }
    });
}

int32_t ihtb_geno_decode(const ihtb_geno* g, int64_t i0, int64_t i1, int64_t j0, int64_t j1, double* out) {
    return guard([&] {
        IHTB_CHECK(g && out, IHTB_EINVAL, "NULL argument");
        IHTB_CHECK(0 <= i0 && i0 <= i1 && i1 <= g->n && 0 <= j0 && j0 <= j1 && j1 <= g->p, IHTB_EDIM,
                   "decode block out of bounds");
        geno_require_ready(g);
        IHTB_CUDA(cudaSetDevice(g->device));
        int64_t total = (i1 - i0) * (j1 - j0);
        if (total == 0) return;
        DBuf<double> d((size_t)total);
        if (geno_is_dense(g)) dense_decode_block(g, i0, i1, j0, j1, d.p);
        else IHTB_LAUNCH(k_decode, (unsigned)ceil_div(total, 256), 256, 0, 0, geno_view(g), g->center, i0, i1, j0, j1, d.p);
        IHTB_CUDA(cudaMemcpy(out, d.p, total * sizeof(double), cudaMemcpyDeviceToHost));
    });
}

int32_t ihtb_geno_packed(const ihtb_geno* g, int64_t j0, int64_t j1, uint8_t* out) {
    return guard([&] {
        IHTB_CHECK(g && out, IHTB_EINVAL, "NULL argument");
        IHTB_CHECK(!geno_is_dense(g), IHTB_EUNSUPPORTED, "a dense handle has no packed genotypes");
        IHTB_CHECK(0 <= j0 && j0 <= j1 && j1 <= g->p, IHTB_EDIM, "column range out of bounds");
        geno_require_ready(g);
        IHTB_CUDA(cudaSetDevice(g->device));
        if (j1 == j0) return;
        int64_t cols_per = (int64_t(256) << 20) / g->nbytes;
        if (cols_per < 1) cols_per = 1;
        if (cols_per > j1 - j0) cols_per = j1 - j0;
        DBuf<uint8_t> staging((size_t)(cols_per * g->nbytes));
        for (int64_t j = j0; j < j1; j += cols_per) {
            int64_t h = (j1 - j < cols_per) ? j1 - j : cols_per;
            IHTB_LAUNCH(k_export, (unsigned)ceil_div(h * g->nbytes, 256), 256, 0, 0, geno_view(g), j, h, staging.p);
            IHTB_CUDA(cudaMemcpy(out + (j - j0) * g->nbytes, staging.p, (size_t)(h * g->nbytes),
                                 cudaMemcpyDeviceToHost));
        }
    });
}

// raw bytes of the ternary copy, exactly as they lie in HBM (tests pin the format against a host twin, synth.ternary_tiles)
int32_t ihtb_geno_ternary_tiles(const ihtb_geno* g, uint8_t* out, int64_t out_bytes) {
    return guard([&] {
        IHTB_CHECK(g && out, IHTB_EINVAL, "NULL argument");
        IHTB_CHECK(!geno_is_dense(g), IHTB_EUNSUPPORTED, "a dense handle has no ternary copy");
        geno_require_ready(g);
        IHTB_CHECK(g->tern.p != nullptr, IHTB_EINVAL, "this handle holds no ternary copy");
        const int64_t bytes = g->tern_slabs * g->p4 * 128;
        IHTB_CHECK(out_bytes == bytes, IHTB_EDIM, "the ternary copy has " + std::to_string(bytes) + " bytes");
        IHTB_CUDA(cudaSetDevice(g->device));
        IHTB_CUDA(cudaMemcpy(out, g->tern.p, (size_t)bytes, cudaMemcpyDeviceToHost));
    });
}

int32_t ihtb_geno_destroy(ihtb_geno* g) {
    return guard([&] {
        if (g) {
            cudaSetDevice(g->device);
            ihtb_internal_fit_cache_clear(g->device);   // parked fit workspaces give their memory back with the matrix
            delete g;
        }
    });
}

}  // extern "C"
