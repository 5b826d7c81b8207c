// Multivariate-Normal IHT (BASELINE config 4): the mIHTVariable loop of the reference on the device.
//
// Reference function (src/multivariate.jl) -> here
//   init_iht_indices! :376-452 -> ihtb_mvfit::init          loglikelihood :9-13, solve_Sigma! :276-282 -> resid_gram + host r x r
//   update_xb! :21-31, update_mu! :39-43, update_resid! :50-58 -> k_x_support<M> + k_mv_resid_gram
//   score!/update_df! :66-92 (skinny X'R, SnpArrays.mul! with an n x r matrix at :85) -> k_mv_score + the sweep:
//       sweep_mode PAIR reads the matrix once per TWO traits (half2 lookup tables, sweep_lut.cu), an odd last trait and
//       sweep_mode FAST / EXACT take one single-vector pass per trait; every candidate entry is re-scored in FP64
//   iht_stepsize! :220-254 (pivoted Cholesky, permutation dropped) -> k_x_support<M> + k_mv_stepsize + host dpstrf
//   _iht_gradstep!/project_k! :99-127 -> topk_candidates over the r*p entries + exact re-scoring + host top-k
//   save_prev! :356-367, check_convergence :454-458, backtrack! :460-473, save_best_model! :485-496, pve src/pve.jl:35
// Layout: traits are columns of n x r column-major device arrays (the reference stores r x n); B is kept k-sparse on
// the host keyed by (column j, trait t); results are written trait-fastest like Julia's r x p matrices.
// Restriction: every covariate is kept (zkeep all true) -- with a false entry the reference's matrix unvectorize!
// (:172-189) reads the wrong slice, so there is no behaviour to reproduce.
#include "glm.cuh"
#include "topk.cuh"
#include "comm.cuh"
#include <algorithm>
#include <chrono>
#include <cmath>
#include <map>
#include <memory>

namespace ihtb {
void sweep_xt_v_with_means(const ihtb_geno* g, const double* dV, const double* vbar_host, int64_t m, double* dOut,
                           int mode, cudaStream_t s, void* scratch_any, float* sweep_ms, double* d_l2 = nullptr,
                           const TopkFuse* tf = nullptr);
void* sweep_scratch_create();
void sweep_scratch_destroy(void* p);
void sweep_class_sums(const ihtb_geno* g, const double* d_v, double* d_w1, double* d_w2, double* d_wm, cudaStream_t s,
                      void* scratch_any);

constexpr int MV_MAXR = 20;       // the reference paper goes up to 18 traits
constexpr int MV_THREADS = 256;
static inline int mv_grid(int64_t n) {
    int64_t b = ceil_div(n, MV_THREADS);
    return (int)(b < 1 ? 1 : (b > GLM_MAX_BLOCKS ? GLM_MAX_BLOCKS : b));
}
struct MvSmall { double a[MV_MAXR * MV_MAXR]; };   // an r x r matrix passed by value (row-major a[i*r + j])

// mu = BX + Z C', resid = (Y - mu) w ; partial sums: Gram[i][j] = sum resid_i resid_j (r*r), then sum w
__global__ void __launch_bounds__(MV_THREADS)
k_mv_resid_gram(int64_t n, int r, int64_t q, const double* __restrict__ BX, const double* __restrict__ Z,
                const double* __restrict__ C /*r x q row-major*/, const double* __restrict__ Y,
                const double* __restrict__ w, double* __restrict__ mu, double* __restrict__ resid,
                double* __restrict__ part) {
    __shared__ double sh[32];
    double g[MV_MAXR * (MV_MAXR + 1) / 2];
    const int ng = r * (r + 1) / 2;
    for (int e = 0; e < ng; ++e) g[e] = 0.0;
    double sw = 0.0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double rs[MV_MAXR];
        const double wi = w[i];
        for (int t = 0; t < r; ++t) {
            double cz = 0.0;
            for (int64_t l = 0; l < q; ++l) cz += C[t * q + l] * Z[i + l * n];
            double m = BX[i + (int64_t)t * n] + cz;
            mu[i + (int64_t)t * n] = m;
            rs[t] = (Y[i + (int64_t)t * n] - m) * wi;
            resid[i + (int64_t)t * n] = rs[t];
        }
        int e = 0;
        for (int a = 0; a < r; ++a)
            for (int b = a; b < r; ++b) g[e++] += rs[a] * rs[b];
        sw += wi;
    }
    const int nv = ng + 1;
    for (int e = 0; e < ng; ++e) {
        double v = block_sum(g[e], sh);
        if (threadIdx.x == 0) part[blockIdx.x * nv + e] = v;
    }
    double v = block_sum(sw, sh);
    if (threadIdx.x == 0) part[blockIdx.x * nv + ng] = v;
}

// R1 = resid * Gamma' (per sample: Gamma * resid_i); partial sums: [0,r) sum R1_t, [r,2r) sum |R1_t|, then df2[t][l]
__global__ void __launch_bounds__(MV_THREADS)
k_mv_score(int64_t n, int r, int64_t q, const double* __restrict__ resid, MvSmall G, const double* __restrict__ Z,
           double* __restrict__ R1, double* __restrict__ part) {
    __shared__ double sh[32];
    double s1[MV_MAXR], sa[MV_MAXR];
    for (int t = 0; t < r; ++t) { s1[t] = 0.0; sa[t] = 0.0; }
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double rs[MV_MAXR];
        for (int t = 0; t < r; ++t) rs[t] = resid[i + (int64_t)t * n];
        for (int t = 0; t < r; ++t) {
            double v = 0.0;
            for (int u = 0; u < r; ++u) v += G.a[t * r + u] * rs[u];
            R1[i + (int64_t)t * n] = v;
            s1[t] += v; sa[t] += fabs(v);
        }
    }
    const int nv = 2 * r + r * (int)q;
    for (int t = 0; t < r; ++t) {
        double v = block_sum(s1[t], sh);
        if (threadIdx.x == 0) part[blockIdx.x * nv + t] = v;
        v = block_sum(sa[t], sh);
        if (threadIdx.x == 0) part[blockIdx.x * nv + r + t] = v;
    }
    for (int t = 0; t < r; ++t)
        for (int64_t l = 0; l < q; ++l) {
            double a = 0.0;
            for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
                a += R1[i + (int64_t)t * n] * Z[i + l * n];
            a = block_sum(a, sh);
            if (threadIdx.x == 0) part[blockIdx.x * nv + 2 * r + t * (int)q + (int)l] = a;
        }
}

// denom = sum_i || U (V_i w_i) ||^2
__global__ void __launch_bounds__(MV_THREADS)
k_mv_stepsize(int64_t n, int r, const double* __restrict__ V, const double* __restrict__ w, MvSmall U,
              double* __restrict__ part) {
    __shared__ double sh[32];
    double a = 0.0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double v[MV_MAXR];
        const double wi = w[i];
        for (int t = 0; t < r; ++t) v[t] = V[i + (int64_t)t * n] * wi;
        for (int t = 0; t < r; ++t) {
            double s = 0.0;
            for (int u = 0; u < r; ++u) s += U.a[t * r + u] * v[u];
            a += s * s;
        }
    }
    a = block_sum(a, sh);
    if (threadIdx.x == 0) part[blockIdx.x] = a;
}

// per trait: partial sums [t] sum mu_t, [r+t] sum y_t ; and second pass sums of squares about the means
__global__ void __launch_bounds__(MV_THREADS)
k_mv_moments(int64_t n, int r, const double* __restrict__ mu, const double* __restrict__ Y, MvSmall means, int pass,
             double* __restrict__ part) {
    __shared__ double sh[32];
    for (int t = 0; t < r; ++t) {
        double a = 0.0, b = 0.0;
        for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
            double m = mu[i + (int64_t)t * n], y = Y[i + (int64_t)t * n];
            if (pass == 0) { a += m; b += y; }
            else { double dm = m - means.a[t], dy = y - means.a[r + t]; a += dm * dm; b += dy * dy; }
        }
        a = block_sum(a, sh); b = block_sum(b, sh);
        if (threadIdx.x == 0) { part[blockIdx.x * 2 * r + t] = a; part[blockIdx.x * 2 * r + r + t] = b; }
    }
}

__global__ void k_mv_finalize(const double* __restrict__ part, int nblocks, int nv, double* __restrict__ out) {
    int v = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (v >= nv) return;
    double a = 0.0;
    for (int b = lane; b < nblocks; b += 32) a += part[b * nv + v];
    a = warp_sum(a);
    if (lane == 0) out[v] = a;
}
__global__ void k_mv_means(const double* __restrict__ scal, int r, int64_t n, double* __restrict__ out) {
    int t = threadIdx.x;
    if (t < r) out[t] = scal[t] / (double)n;
}
__global__ void k_mv_weights(int64_t n, const uint8_t* __restrict__ mask, double* __restrict__ w) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) w[i] = (mask == nullptr || mask[i]) ? 1.0 : 0.0;
}

// ---- r x r host linear algebra ---------------------------------------------------------------------------------
static bool chol_lower(int r, const double* a, double* l) {   // a = l l', row-major
    std::fill(l, l + r * r, 0.0);
    for (int j = 0; j < r; ++j) {
        double d = a[j * r + j];
        for (int k = 0; k < j; ++k) d -= l[j * r + k] * l[j * r + k];
        if (!(d > 0.0)) return false;
        l[j * r + j] = std::sqrt(d);
        for (int i = j + 1; i < r; ++i) {
            double s = a[i * r + j];
            for (int k = 0; k < j; ++k) s -= l[i * r + k] * l[j * r + k];
            l[i * r + j] = s / l[j * r + j];
        }
    }
    return true;
}
static void spd_inverse(int r, const double* l, double* inv) {   // (l l')^-1 from the lower factor
    std::vector<double> li((size_t)r * r, 0.0);
    for (int i = 0; i < r; ++i) {
        li[i * r + i] = 1.0 / l[i * r + i];
        for (int j = 0; j < i; ++j) {
            double s = 0.0;
            for (int k = j; k < i; ++k) s -= l[i * r + k] * li[k * r + j];
            li[i * r + j] = s / l[i * r + i];
        }
    }
    for (int i = 0; i < r; ++i)
        for (int j = 0; j < r; ++j) {
            double s = 0.0;
            for (int k = std::max(i, j); k < r; ++k) s += li[k * r + i] * li[k * r + j];
            inv[i * r + j] = s;
        }
}
// LAPACK dpstrf(uplo='U') order: largest remaining diagonal first (first maximum wins); returns U, permutation dropped
static bool pivoted_chol_upper(int r, const double* a_in, double* u) {
    std::vector<double> s(a_in, a_in + r * r);
    for (int i = 0; i < r; ++i)
        for (int j = 0; j < i; ++j) s[i * r + j] = s[j * r + i];      // Symmetric(A, :U)
    std::fill(u, u + r * r, 0.0);
    for (int j = 0; j < r; ++j) {
        int pvt = j;
        for (int i = j + 1; i < r; ++i)
            if (s[i * r + i] > s[pvt * r + pvt]) pvt = i;
        if (pvt != j) {
            for (int c = 0; c < r; ++c) std::swap(s[j * r + c], s[pvt * r + c]);
            for (int c = 0; c < r; ++c) std::swap(s[c * r + j], s[c * r + pvt]);
            for (int c = 0; c < r; ++c) std::swap(u[c * r + j], u[c * r + pvt]);
        }
        double ajj = s[j * r + j];
        if (!(ajj > 0.0)) return false;
        ajj = std::sqrt(ajj);
        u[j * r + j] = ajj;
        for (int c = j + 1; c < r; ++c) u[j * r + c] = s[j * r + c] / ajj;
        for (int a = j + 1; a < r; ++a)
            for (int b = j + 1; b < r; ++b) s[a * r + b] -= u[j * r + a] * u[j * r + b];
    }
    return true;
}

}  // namespace ihtb

using namespace ihtb;

static const double kFastBoundMv = 1.0 / 262144.0;
static const double kExactBoundMv = 1e-13;
// sweep_mode PAIR: every bound is an L2 bound over the handle's sgn scale (fit.cu kPairBound): paired traits
// 3.1 * 2^-11 ||u||_2 sgn_j (half2 tables), an odd last trait 2^-20 ||u||_2 sgn_j (FP32 tables: 12 roundings of 2^-24)
static const double kPairBoundMv = 3.1 / 2048.0;
static const double kFastL2BoundMv = 1.0 / 1048576.0;

struct ihtb_mvfit {
    const ihtb_geno* g = nullptr;
    int device = 0;
    int64_t n = 0, p = 0, q = 0;          // p = local SNP columns
    int r = 0;
    // SNP-sharded fits (like fit.cu): this rank owns global columns [j0, j0 + p); Y, Z, every n x r array and the
    // k-sparse model (keyed by GLOBAL position j*r + t) are replicated; partial BX / V products are all-reduced, exact
    // gradient entries and candidate columns are exchanged over the communicator's peer-memory collectives
    ihtb_comm* comm = nullptr;
    int64_t j0 = 0, p_global = 0;
    DBuf<int64_t> d_xch, d_xchall;        // candidate-column exchange block [count | cols[cap]] and its gathered copy
    HBuf<int64_t> h_xchall;
    bool is_local(int64_t j) const { return j >= j0 && j < j0 + p; }
    ihtb_cfg cfg{};
    cudaStream_t s = nullptr;
    int cap = 4096;
    DBuf<double> d_Y, d_Z, d_w, d_BX, d_mu, d_resid, d_R1, d_V, d_dfa, d_b0d, d_part, d_scal, d_C, d_coef, d_gout,
        d_vbar, d_sval, d_bounds, d_sinvrep;
    DBuf<uint8_t> d_mask;
    DBuf<uint32_t> d_keyL, d_keyU;
    DBuf<int> d_hist;
    DBuf<int64_t> d_sel, d_idx, d_cols, d_sidx;
    HBuf<double> h_scal, h_gout, h_l2;
    DBuf<double> d_l2;                               // ||R1_t - mean||_2 per trait (PAIR sweeps: L2 error bounds)
    HBuf<int64_t> h_sel;
    void* sweep_scratch = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    TopkCtx tk{};

    // host model: entries keyed by position in vec(B) = j*r + t (Julia's column-major r x p order)
    std::map<int64_t, double> B, B0, bestB;
    std::vector<double> C, C0, bestC, df2;           // r x q row-major
    std::vector<double> Gamma, Gamma0;               // r x r row-major
    std::map<int64_t, std::vector<double>> df_exact; // column -> r exact gradient entries
    std::map<int64_t, double> dfs;                   // sparse (projected) df after init, keyed like B
    bool df_sparse = false, inited = false;
    std::vector<double> bounds;                      // per-trait sweep error bound
    std::vector<int64_t> b0d_pos;
    double n_train = 0.0;
    std::vector<double> pve;
    int64_t n_sweeps = 0, n_backtracks = 0, n_cand_iter = 0;
    double sweep_ms_total = 0.0;

    ~ihtb_mvfit() {
        if (sweep_scratch) sweep_scratch_destroy(sweep_scratch);
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        if (s) cudaStreamDestroy(s);
    }
    void sync() { IHTB_CUDA(cudaStreamSynchronize(s)); }
    template <typename T>
    void upload(T* dst, const T* src, size_t count) {
        if (count) IHTB_CUDA(cudaMemcpyAsync(dst, src, count * sizeof(T), cudaMemcpyHostToDevice, s));
    }
    void finalize(int grid, int nv) {
        IHTB_LAUNCH(k_mv_finalize, (unsigned)ceil_div(nv, 4), 128, 0, s, d_part.p, grid, nv, d_scal.p);
    }
    void readback(int nv) {
        IHTB_CUDA(cudaMemcpyAsync(h_scal.p, d_scal.p, nv * sizeof(double), cudaMemcpyDeviceToHost, s));
        sync();
    }
    // host wall-clock per phase (every phase ends in a readback, so these are device-inclusive); IHTB_MV_TIMING=1 prints them
    double phase_s[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // 5..7: inside gradstep (top-k, exchange, exact re-scoring)
    template <typename F>
    auto timed(int ph, F&& fn) {
        auto t0 = std::chrono::steady_clock::now();
        struct Stop {
            double& acc; std::chrono::steady_clock::time_point t0;
            ~Stop() { acc += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count(); }
        } stop{phase_s[ph], t0};
        return fn();
    }
    static std::vector<int64_t> support_cols(const std::map<int64_t, double>& M, int r) {
        std::vector<int64_t> cols;
        for (auto& kv : M)
            if (kv.second != 0.0 && (cols.empty() || cols.back() != kv.first / r)) cols.push_back(kv.first / r);
        return cols;
    }
    MvSmall small(const std::vector<double>& m) const {
        MvSmall o;
        std::fill(o.a, o.a + MV_MAXR * MV_MAXR, 0.0);
        std::copy(m.begin(), m.end(), o.a);
        return o;
    }

    // d_out (n x r) = sum_{j in cols} x[:, j] * coef[j][t]   (update_xb! :21-31 / iht_stepsize! :234)
    void support_matmat(const std::vector<int64_t>& cols, const std::vector<double>& coef /*|cols| x r col-major*/,
                        double* d_out) {
        // this rank's columns (all of them without a communicator), local indices, same order
        std::vector<int64_t> loc; std::vector<size_t> src;
        for (size_t c = 0; c < cols.size(); ++c)
            if (is_local(cols[c])) { loc.push_back(cols[c] - j0); src.push_back(c); }
        if (loc.empty()) {
            IHTB_CUDA(cudaMemsetAsync(d_out, 0, n * r * sizeof(double), s));
        } else {
            std::vector<double> cl(loc.size() * (size_t)r);
            for (int t = 0; t < r; ++t)
                for (size_t c = 0; c < loc.size(); ++c) cl[c + (size_t)t * loc.size()] = coef[src[c] + (size_t)t * cols.size()];
            upload(d_idx.p, loc.data(), loc.size());
            upload(d_coef.p, cl.data(), cl.size());
            x_support(g, d_idx.p, (int64_t)loc.size(), d_coef.p, r, d_out, s);
        }
        if (comm) comm_allreduce_sum_f64(comm, d_out, (size_t)(n * r), s);
    }
    void update_xb() {
        std::vector<int64_t> cols = support_cols(B, r);
        std::vector<double> coef(cols.size() * r, 0.0);
        for (size_t c = 0; c < cols.size(); ++c)
            for (int t = 0; t < r; ++t) {
                auto it = B.find(cols[c] * r + t);
                if (it != B.end()) coef[c + (size_t)t * cols.size()] = it->second;
            }
        support_matmat(cols, coef, d_BX.p);
    }
    // update_mu!, update_resid!, Gram = resid resid' (r x r, host copy)
    std::vector<double> resid_gram() {
        upload(d_C.p, C.data(), C.size());
        int grid = mv_grid(n);
        int ng = r * (r + 1) / 2;
        IHTB_LAUNCH(k_mv_resid_gram, grid, MV_THREADS, 0, s, n, r, q, d_BX.p, d_Z.p, d_C.p, d_Y.p, d_w.p, d_mu.p,
                    d_resid.p, d_part.p);
        finalize(grid, ng + 1);
        readback(ng + 1);
        std::vector<double> G((size_t)r * r);
        int e = 0;
        for (int a = 0; a < r; ++a)
            for (int b = a; b < r; ++b) { G[a * r + b] = h_scal.p[e]; G[b * r + a] = h_scal.p[e]; ++e; }
        n_train = h_scal.p[ng];
        return G;
    }
    // solve_Sigma! :276-282 followed by loglikelihood :9-13 (the Gram matrix is the same in both)
    double solve_sigma_and_logl() {
        std::vector<double> G = resid_gram();
        std::vector<double> S((size_t)r * r), L((size_t)r * r);
        for (int e = 0; e < r * r; ++e) S[e] = G[e] / n_train;
        if (!chol_lower(r, S.data(), L.data())) return NAN;
        spd_inverse(r, L.data(), Gamma.data());
        double logdet = 0.0;
        for (int i = 0; i < r; ++i) logdet -= 2.0 * std::log(L[i * r + i]);      // logdet(Gamma) = -logdet(Sigma)
        double tr = 0.0;
        for (int i = 0; i < r; ++i)
            for (int j = 0; j < r; ++j) tr += Gamma[i * r + j] * G[j * r + i];
        return n_train / 2.0 * logdet - 0.5 * tr;
    }
    void exact_df(const std::vector<int64_t>& cols) {
        std::vector<int64_t> need;
        for (int64_t j : cols)
            if (!df_exact.count(j)) need.push_back(j);
        if (need.empty()) return;
        IHTB_CHECK(need.size() * r <= d_gout.n && need.size() <= d_cols.n, IHTB_ENUMERIC, "too many columns to re-score");
        // columns of other shards are marked -1: the kernel writes 0 for them and the all-reduce fills them in
        std::vector<int64_t> loc(need.size());
        for (size_t c = 0; c < need.size(); ++c) loc[c] = is_local(need[c]) ? need[c] - j0 : -1;
        upload(d_cols.p, loc.data(), loc.size());
        xt_gather(g, d_cols.p, (int64_t)need.size(), d_R1.p, r, d_vbar.p, d_gout.p, s);
        if (comm) comm_allreduce_sum_f64(comm, d_gout.p, need.size() * (size_t)r, s);
        IHTB_CUDA(cudaMemcpyAsync(h_gout.p, d_gout.p, need.size() * r * sizeof(double), cudaMemcpyDeviceToHost, s));
        sync();
        for (size_t c = 0; c < need.size(); ++c) {
            std::vector<double> v((size_t)r);
            for (int t = 0; t < r; ++t) v[t] = h_gout.p[c + (size_t)t * need.size()];
            df_exact[need[c]] = v;
        }
        n_cand_iter += (int64_t)need.size();
    }
    // score! :66-92
    void score_and_sweep() {
        int grid = mv_grid(n);
        int nv = 2 * r + r * (int)q;
        IHTB_LAUNCH(k_mv_score, grid, MV_THREADS, 0, s, n, r, q, d_resid.p, small(Gamma), d_Z.p, d_R1.p, d_part.p);
        finalize(grid, nv);
        IHTB_LAUNCH(k_mv_means, 1, 32, 0, s, d_scal.p, r, n, d_vbar.p);
        IHTB_CUDA(cudaMemcpyAsync(h_scal.p, d_scal.p, nv * sizeof(double), cudaMemcpyDeviceToHost, s));
        IHTB_CUDA(cudaEventRecord(ev0, s));
        const bool l2mode = cfg.sweep_mode == IHTB_SWEEP_PAIR;
        if (l2mode && d_l2.n < (size_t)r) { d_l2.alloc((size_t)r); h_l2.alloc((size_t)r); }
        sweep_xt_v_with_means(g, d_R1.p, d_vbar.p, r, d_dfa.p, cfg.sweep_mode, s, sweep_scratch, nullptr,
                              l2mode ? d_l2.p : nullptr);
        IHTB_CUDA(cudaEventRecord(ev1, s));
        if (l2mode) IHTB_CUDA(cudaMemcpyAsync(h_l2.p, d_l2.p, (size_t)r * sizeof(double), cudaMemcpyDeviceToHost, s));
        n_sweeps += r;
        df_exact.clear();
        df_sparse = false;
        std::vector<int64_t> cols = support_cols(B, r);
        if (!cols.empty()) exact_df(cols); else sync();
        float ms = 0.f;
        IHTB_CUDA(cudaEventElapsedTime(&ms, ev0, ev1));
        sweep_ms_total += ms;
        for (int t = 0; t < r; ++t) {
            double mean = h_scal.p[t] / (double)n;
            double ul1 = h_scal.p[r + t] + (double)n * std::fabs(mean);
            if (l2mode) bounds[t] = (t < 2 * (r / 2) ? kPairBoundMv : kFastL2BoundMv) * h_l2.p[t];
            else bounds[t] = (cfg.sweep_mode == IHTB_SWEEP_EXACT ? kExactBoundMv : kFastBoundMv) * ul1;
        }
        for (int e = 0; e < r * (int)q; ++e) df2[e] = h_scal.p[2 * r + e];
    }
    double df_entry(int64_t pos) const {
        if (df_sparse) {
            auto it = dfs.find(pos);
            return it == dfs.end() ? 0.0 : it->second;
        }
        return df_exact.at(pos / r)[pos % r];
    }
    // iht_stepsize! :220-254
    double stepsize() {
        std::vector<int64_t> cols = support_cols(B, r);
        if (df_sparse) cols = support_cols(dfs, r);
        std::vector<double> coef(cols.size() * r, 0.0);
        double numer = 0.0;
        for (size_t c = 0; c < cols.size(); ++c)
            for (int t = 0; t < r; ++t) {
                double v = df_entry(cols[c] * r + t);
                coef[c + (size_t)t * cols.size()] = v;
                numer += v * v;
            }
        support_matmat(cols, coef, d_V.p);
        std::vector<double> U((size_t)r * r);
        IHTB_CHECK(pivoted_chol_upper(r, Gamma.data(), U.data()), IHTB_ENUMERIC,
                   "RankDeficientException in the pivoted Cholesky of the precision matrix");
        Gamma = U;     // the reference overwrites Gamma with the factor; solve_Sigma! rebuilds it after the step
        int grid = mv_grid(n);
        IHTB_LAUNCH(k_mv_stepsize, grid, MV_THREADS, 0, s, n, r, d_V.p, d_w.p, small(U), d_part.p);
        finalize(grid, 1);
        readback(1);
        double eta = numer / h_scal.p[0];
        if (std::isinf(eta) || std::isnan(eta)) eta = 1e-8;
        return eta;
    }
    void sync_b0d() {
        if (!b0d_pos.empty()) {
            upload(d_sidx.p, b0d_pos.data(), b0d_pos.size());
            scatter_dense(d_b0d.p, d_sidx.p, nullptr, (int64_t)b0d_pos.size(), 1, s);
        }
        b0d_pos.clear();
        std::vector<double> vals;
        for (auto& kv : B0)
            if (kv.second != 0.0 && is_local(kv.first / r)) {   // device vector is trait-major over LOCAL columns: e = t*p + (j - j0)
                b0d_pos.push_back((kv.first % r) * p + (kv.first / r - j0));
                vals.push_back(kv.second);
            }
        if (!b0d_pos.empty()) {
            upload(d_sidx.p, b0d_pos.data(), b0d_pos.size());
            upload(d_sval.p, vals.data(), vals.size());
            scatter_dense(d_b0d.p, d_sidx.p, d_sval.p, (int64_t)b0d_pos.size(), 0, s);
        }
    }
    // candidate columns of the top-k over the r*p entries |B0 + eta*df|
    std::vector<int64_t> device_candidate_cols(double eta) {
        std::vector<int64_t> cols = timed(5, [&] { return local_candidate_cols(eta); });
        if (!comm) return cols;
        return timed(6, [&] { return exchange_candidate_cols(cols); });
    }
    std::vector<int64_t> local_candidate_cols(double eta) {
        upload(d_bounds.p, bounds.data(), (size_t)r);
        topk_candidates_blocked(tk, d_dfa.p, d_b0d.p,
                                cfg.sweep_mode == IHTB_SWEEP_PAIR ? g->sgn.p : g->sinv.p, p,
                                d_bounds.p, eta, cfg.k, s);
        IHTB_CUDA(cudaMemcpyAsync(h_sel.p, d_sel.p, (2 + cap) * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
        sync();
        const TopkState* st = reinterpret_cast<const TopkState*>(h_sel.p);
        IHTB_CHECK(st->count <= cap, IHTB_ENUMERIC, "degenerate projection: too many entries within the error bound");
        std::vector<int64_t> cols;
        for (int t = 0; t < st->count; ++t) cols.push_back(h_sel.p[2 + t] % p + j0);
        return cols;
    }
    std::vector<int64_t> exchange_candidate_cols(std::vector<int64_t> cols) {
        // the selection ran over all shards' entries (histograms all-reduced, topk.cu): every rank holds exactly its part
        // of the candidate set a single device would find; one all-gather of fixed blocks [count | global columns]
        const size_t blk = 1 + (size_t)cap;
        std::vector<int64_t> mine(blk, -1);
        mine[0] = (int64_t)cols.size();
        std::copy(cols.begin(), cols.end(), mine.begin() + 1);
        upload(d_xch.p, mine.data(), blk);
        comm_allgather_i64(comm, d_xch.p, d_xchall.p, blk, s);
        IHTB_CUDA(cudaMemcpyAsync(h_xchall.p, d_xchall.p, (size_t)comm->nranks * blk * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
        sync();
        cols.clear();
        for (int rk = 0; rk < comm->nranks; ++rk) {
            const int64_t* b_ = h_xchall.p + (size_t)rk * blk;
            cols.insert(cols.end(), b_ + 1, b_ + 1 + b_[0]);
        }
        return cols;
    }
    // _iht_gradstep! / project_k! :99-127 (all covariates kept: only entries of B compete for the k slots)
    void gradstep(double eta) {
        std::vector<int64_t> cols;
        if (df_sparse) {
            cols = support_cols(dfs, r);
        } else {
            cols = device_candidate_cols(eta);
        }
        for (auto& kv : B0) cols.push_back(kv.first / r);
        std::sort(cols.begin(), cols.end());
        cols.erase(std::unique(cols.begin(), cols.end()), cols.end());
        if (!df_sparse) timed(7, [&] { exact_df(cols); return 0; });
        struct Item { double a; int64_t pos; double v; };
        std::vector<Item> items;
        for (int64_t j : cols)
            for (int t = 0; t < r; ++t) {
                int64_t pos = j * r + t;
                auto it = B0.find(pos);
                double v = (it == B0.end() ? 0.0 : it->second) + eta * df_entry(pos);
                items.push_back({std::fabs(v), pos, v});
            }
        std::sort(items.begin(), items.end(), [](const Item& x, const Item& y) {
            return x.a > y.a || (x.a == y.a && x.pos < y.pos);
        });
        B.clear();
        for (size_t t = 0; t < items.size() && (int64_t)t < cfg.k; ++t)
            if (items[t].v != 0.0) B[items[t].pos] = items[t].v;
        for (size_t e = 0; e < C.size(); ++e) C[e] = C0[e] + eta * df2[e];
    }
    double save_prev(double cur, double best) {
        B0 = B; C0 = C; Gamma0 = Gamma;
        if (cur > best) { bestB = B; bestC = C; }
        sync_b0d();
        return std::max(cur, best);
    }
    double check_convergence() const {
        double nrm = 0.0, b0max = 0.0;
        for (auto& kv : B) {
            auto it = B0.find(kv.first);
            nrm = std::max(nrm, std::fabs(kv.second - (it == B0.end() ? 0.0 : it->second)));
        }
        for (auto& kv : B0) {
            if (!B.count(kv.first)) nrm = std::max(nrm, std::fabs(kv.second));
            b0max = std::max(b0max, std::fabs(kv.second));
        }
        for (size_t e = 0; e < C.size(); ++e) {
            nrm = std::max(nrm, std::fabs(C[e] - C0[e]));
            b0max = std::max(b0max, std::fabs(C0[e]));
        }
        return nrm / (b0max + 1.0);
    }
    void save_best_model() {
        B = bestB; C = bestC;
        update_xb();
        resid_gram();     // mu = BX + CZ with the best model
    }
    void compute_pve() {
        int grid = mv_grid(n);
        MvSmall means = small(std::vector<double>());
        IHTB_LAUNCH(k_mv_moments, grid, MV_THREADS, 0, s, n, r, d_mu.p, d_Y.p, means, 0, d_part.p);
        finalize(grid, 2 * r);
        readback(2 * r);
        for (int t = 0; t < 2 * r; ++t) means.a[t] = h_scal.p[t] / (double)n;
        IHTB_LAUNCH(k_mv_moments, grid, MV_THREADS, 0, s, n, r, d_mu.p, d_Y.p, means, 1, d_part.p);
        finalize(grid, 2 * r);
        readback(2 * r);
        pve.assign((size_t)r, 0.0);
        for (int t = 0; t < r; ++t) pve[t] = h_scal.p[t] / h_scal.p[r + t];
    }
    void set_weights(const uint8_t* mask) {
        const uint8_t* dm = nullptr;
        if (mask) { upload(d_mask.p, mask, (size_t)n); dm = d_mask.p; }
        IHTB_LAUNCH(k_mv_weights, (unsigned)ceil_div(n, 256), 256, 0, s, n, dm, d_w.p);
    }
    // init_iht_indices! :376-452
    // initialize_beta! (src/multivariate.jl:519-558) + project_k!(v) + update_xb! (:425-429): every B[t, j] starts at
    // the slope of the univariate regression of trait t on [1, x_j] over the training samples (clamped to +-2), the
    // intercept of trait t at the mean of all those regressions' intercepts; then the k largest entries are kept.
    // The per-SNP sums come from the exact class-sum sweep (one pass for the weights, one per trait), like the
    // univariate ihtb_fit_init_beta.  The reference accumulates the intercepts from several threads without
    // synchronisation; this is the single-thread result.
    void do_init_beta(const uint8_t* train_mask, const std::vector<double>& sy) {
        // SNP-sharded fits: class sums and regressions are per column (no communication); the intercept sums are
        // all-reduced and the ranks' local top-k entries of the initial B all-gathered for the global projection
        DBuf<double> cls((size_t)(6 * p)), bd((size_t)(p * r)), wy((size_t)n);
        double *W1 = cls.p, *W2 = W1 + p, *Wm = W2 + p, *Y1 = Wm + p, *Y2 = Y1 + p, *Ym = Y2 + p;
        sweep_class_sums(g, d_w.p, W1, W2, Wm, s, sweep_scratch);
        ++n_sweeps;
        std::vector<double> c0sum((size_t)r, 0.0);
        for (int t = 0; t < r; ++t) {
            GlmCtx tmp{n, q, d_Z.p, d_Y.p + (size_t)t * n, d_w.p, nullptr, nullptr, nullptr, nullptr, d_part.p, d_scal.p,
                       IHTB_NORMAL, IHTB_LINK_IDENTITY, 1.0};
            init_beta_products(tmp, wy.p, s);
            sweep_class_sums(g, wy.p, Y1, Y2, Ym, s, sweep_scratch);
            ++n_sweeps;
            init_beta_solve(tmp, p, W1, W2, Wm, Y1, Y2, Ym, n_train, sy[(size_t)t], g->mu.p, g->sinv.p, g->impute,
                            bd.p + (size_t)t * p, s);
            readback(1);
            c0sum[(size_t)t] = h_scal.p[0];
        }
        if (comm) {
            upload(d_scal.p, c0sum.data(), (size_t)r);
            comm_allreduce_sum_f64(comm, d_scal.p, (size_t)r, s);
            readback(r);
            std::copy(h_scal.p, h_scal.p + r, c0sum.begin());
        }
        // covariates 2..q: the same 2x2 regression on the host (r*q*n work)
        std::fill(C.begin(), C.end(), 0.0);
        if (q > 1) {
            std::vector<double> hY((size_t)(n * r)), hZ((size_t)(n * q));
            IHTB_CUDA(cudaMemcpyAsync(hY.data(), d_Y.p, hY.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
            IHTB_CUDA(cudaMemcpyAsync(hZ.data(), d_Z.p, hZ.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
            sync();
            for (int t = 0; t < r; ++t)
                for (int64_t l = 1; l < q; ++l) {
                    double sx = 0.0, sxx = 0.0, sxy = 0.0;
                    for (int64_t i = 0; i < n; ++i) {
                        if (train_mask && !train_mask[i]) continue;
                        const double z = hZ[(size_t)(i + l * n)];
                        sx += z; sxx += z * z; sxy += z * hY[(size_t)(i + (int64_t)t * n)];
                    }
                    double icpt = sy[(size_t)t], slope = sxy;
                    const double u11 = std::sqrt(n_train), u12 = sx / u11, dd = sxx - u12 * u12;
                    if (n_train > 0 && dd > 0) {
                        const double u22 = std::sqrt(dd), t1 = sy[(size_t)t] / u11, t2 = (sxy - u12 * t1) / u22;
                        slope = t2 / u22; icpt = (t1 - u12 * slope) / u11;
                    }
                    c0sum[(size_t)t] += icpt;
                    C[(size_t)(t * q + l)] = std::min(std::max(slope, -2.0), 2.0);
                }
        }
        for (int t = 0; t < r; ++t)
            C[(size_t)(t * q)] = std::min(std::max(c0sum[(size_t)t] / (double)(p_global + q - 1), -2.0), 2.0);
        // project_k!(v): the k largest |B| entries (ties: lowest position in vec(B)); covariates are all kept
        std::vector<double> zeros((size_t)r, 0.0);
        upload(d_bounds.p, zeros.data(), zeros.size());
        topk_candidates_blocked(tk, bd.p, nullptr, g->sinv.p, p, d_bounds.p, 1.0, cfg.k, s);
        IHTB_CUDA(cudaMemcpyAsync(h_sel.p, d_sel.p, (2 + cap) * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
        sync();
        const TopkState* st = reinterpret_cast<const TopkState*>(h_sel.p);
        IHTB_CHECK(st->count <= cap && (size_t)st->count <= d_gout.n, IHTB_ENUMERIC,
                   "degenerate projection of the initial beta (too many ties)");
        const int cnt = st->count;
        take_values(bd.p, d_sel.p + 2, cnt, d_gout.p, s);
        IHTB_CUDA(cudaMemcpyAsync(h_gout.p, d_gout.p, (size_t)cnt * sizeof(double), cudaMemcpyDeviceToHost, s));
        sync();
        struct Item { double a; int64_t pos; double v; };
        std::vector<Item> items;
        for (int e = 0; e < cnt; ++e) {
            const int64_t pos_dev = h_sel.p[2 + e], t = pos_dev / p, j = pos_dev % p + j0;
            items.push_back({std::fabs(h_gout.p[e]), j * r + t, h_gout.p[e]});
        }
        if (comm) {        // two all-gathers of fixed blocks: [count | positions in vec(B)] and [count | value bits]
            const size_t blk = 1 + (size_t)cap;
            std::vector<int64_t> pos_blk(blk, -1), val_blk(blk, 0);
            pos_blk[0] = val_blk[0] = (int64_t)items.size();
            for (size_t e = 0; e < items.size(); ++e) {
                pos_blk[1 + e] = items[e].pos;
                memcpy(&val_blk[1 + e], &items[e].v, sizeof(double));
            }
            std::vector<int64_t> all_pos((size_t)comm->nranks * blk);
            for (int pass = 0; pass < 2; ++pass) {
                upload(d_xch.p, (pass == 0 ? pos_blk : val_blk).data(), blk);
                comm_allgather_i64(comm, d_xch.p, d_xchall.p, blk, s);
                IHTB_CUDA(cudaMemcpyAsync(h_xchall.p, d_xchall.p, all_pos.size() * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
                sync();
                if (pass == 0) std::copy(h_xchall.p, h_xchall.p + all_pos.size(), all_pos.begin());
            }
            items.clear();
            for (int rk = 0; rk < comm->nranks; ++rk)
                for (int64_t e = 0; e < all_pos[(size_t)rk * blk]; ++e) {
                    double v;
                    memcpy(&v, &h_xchall.p[(size_t)rk * blk + 1 + (size_t)e], sizeof(double));
                    items.push_back({std::fabs(v), all_pos[(size_t)rk * blk + 1 + (size_t)e], v});
                }
        }
        std::sort(items.begin(), items.end(), [](const Item& x, const Item& y) {
            return x.a > y.a || (x.a == y.a && x.pos < y.pos);
        });
        B.clear();
        for (size_t e = 0; e < items.size() && (int64_t)e < cfg.k; ++e)
            if (items[e].v != 0.0) B[items[e].pos] = items[e].v;
        B0 = B; C0 = C;
        update_xb();
    }

    void init(const uint8_t* train_mask, bool init_beta = false) {
        IHTB_CHECK(cfg.k >= 1, IHTB_EINVAL, "Multivariate IHT requires k >= 1!");
        B.clear(); B0.clear(); bestB.clear(); dfs.clear(); df_exact.clear(); df_sparse = false;
        C.assign((size_t)r * q, 0.0); C0 = C; bestC = C; df2.assign((size_t)r * q, 0.0);
        Gamma.assign((size_t)r * r, 0.0);
        for (int i = 0; i < r; ++i) Gamma[i * r + i] = 1.0;
        Gamma0 = Gamma;
        bounds.assign((size_t)r, 0.0);
        sync_b0d();
        set_weights(train_mask);
        IHTB_CUDA(cudaMemsetAsync(d_BX.p, 0, n * r * sizeof(double), s));
        // intercept = weighted mean of each trait: use resid_gram with C = 0 to get sum w, then a moments pass
        // (Y*w summed per trait) -- cheap: reuse k_mv_score on "resid" = Y*w with Gamma = I
        std::vector<double> G0 = resid_gram();                       // C = 0, BX = 0 -> resid = Y w, n_train = sum w
        int grid = mv_grid(n);
        int nv = 2 * r + r * (int)q;
        IHTB_LAUNCH(k_mv_score, grid, MV_THREADS, 0, s, n, r, q, d_resid.p, small(Gamma), d_Z.p, d_R1.p, d_part.p);
        finalize(grid, nv);
        readback(nv);
        std::vector<double> sy((size_t)r);
        for (int t = 0; t < r; ++t) { sy[(size_t)t] = h_scal.p[t]; C[t * q + 0] = h_scal.p[t] / n_train; }   // ybar_t (:415-422)
        resid_gram();                                                // CZ, mu, resid
        if (init_beta) {
            do_init_beta(train_mask, sy);
            resid_gram();                                            // mu, resid of the initialised model
        }
        score_and_sweep();                                           // Gamma = I
        if (init_beta) { inited = true; return; }                    // df keeps the full gradient (:436 `if !init_beta`)
        // first k entries of the gradient by magnitude; df becomes its projection (:436-445)
        std::vector<int64_t> cols = device_candidate_cols(1.0);
        std::sort(cols.begin(), cols.end());
        cols.erase(std::unique(cols.begin(), cols.end()), cols.end());
        exact_df(cols);
        struct Item { double a; int64_t pos; double v; };
        std::vector<Item> items;
        for (int64_t j : cols)
            for (int t = 0; t < r; ++t) {
                double v = df_exact.at(j)[t];
                items.push_back({std::fabs(v), j * r + t, v});
            }
        std::sort(items.begin(), items.end(), [](const Item& x, const Item& y) {
            return x.a > y.a || (x.a == y.a && x.pos < y.pos);
        });
        for (size_t t = 0; t < items.size() && (int64_t)t < cfg.k; ++t)
            if (items[t].v != 0.0) dfs[items[t].pos] = items[t].v;
        df_sparse = true;
        inited = true;
    }
    void one_step(double old_logl, double& eta, int& eta_step, double& new_logl) {
        eta = timed(0, [&] { return stepsize(); });
        timed(1, [&] { gradstep(eta); return 0; });
        timed(2, [&] { update_xb(); return 0; });
        new_logl = timed(3, [&] { return solve_sigma_and_logl(); });
        eta_step = 0;
        while (old_logl > new_logl && eta_step < cfg.max_step) {
            eta /= 2;
            B = B0; C = C0; Gamma = Gamma0;
            timed(1, [&] { gradstep(eta); return 0; });
            timed(2, [&] { update_xb(); return 0; });
            new_logl = timed(3, [&] { return solve_sigma_and_logl(); });
            ++eta_step; ++n_backtracks;
        }
        timed(4, [&] { score_and_sweep(); return 0; });
        IHTB_CHECK(!std::isnan(new_logl), IHTB_ENUMERIC, "Loglikelihood function is NaN, aborting...");
        IHTB_CHECK(!std::isinf(new_logl), IHTB_ENUMERIC, "Loglikelihood function is Inf, aborting...");
    }
    void run(ihtb_result* res, ihtb_iter_trace* trace, int64_t trace_cap) {
        IHTB_CHECK(inited, IHTB_EINVAL, "ihtb_mvfit_init must be called before ihtb_mvfit_run");
        auto t0 = std::chrono::steady_clock::now();
        int64_t launches0 = launch_counter(), mm_iter = 0, n_steps = 0, sweeps0 = n_sweeps;
        double next_logl = -INFINITY, best_logl = -INFINITY, ms0 = sweep_ms_total;
        n_backtracks = 0;
        for (int64_t iter = 1; iter <= cfg.max_iter; ++iter) {
            if (iter >= cfg.max_iter) {
                best_logl = save_prev(next_logl, best_logl); save_best_model(); mm_iter = iter;
                break;
            }
            best_logl = save_prev(next_logl, best_logl);
            double eta; int eta_step;
            n_cand_iter = 0;
            one_step(next_logl, eta, eta_step, next_logl);
            ++n_steps;
            double scaled = check_convergence();
            if (trace && iter - 1 < trace_cap)
                trace[iter - 1] = ihtb_iter_trace{next_logl, scaled, eta, eta_step, (int32_t)n_cand_iter};
            if (iter >= cfg.min_iter && scaled < cfg.tol) {
                best_logl = save_prev(next_logl, best_logl); save_best_model(); mm_iter = iter;
                break;
            }
        }
        compute_pve();
        inited = false;
        if (getenv("IHTB_MV_TIMING") && (!comm || comm->rank == 0))
            fprintf(stderr, "[mvfit] %lld steps: stepsize %.3f ms, gradstep %.3f ms, update_xb %.3f ms, sigma/logl %.3f ms, "
                    "score+sweep %.3f ms (sweep kernels %.3f ms); inside gradstep: top-k %.3f, exchange %.3f, re-scoring %.3f ms\n",
                    (long long)n_steps, phase_s[0] * 1e3, phase_s[1] * 1e3, phase_s[2] * 1e3, phase_s[3] * 1e3, phase_s[4] * 1e3,
                    sweep_ms_total - ms0, phase_s[5] * 1e3, phase_s[6] * 1e3, phase_s[7] * 1e3);
        if (res) {
            res->time = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
            res->logl = best_logl; res->iter = mm_iter; res->sigma_g = pve.empty() ? 0.0 : pve[0];
            res->n_sweeps = n_sweeps - sweeps0 + r; res->n_backtracks = n_backtracks;
            res->sweep_seconds = (sweep_ms_total - ms0) * 1e-3;
            res->n_launches = launch_counter() - launches0; res->n_steps = n_steps;
        }
    }
};

extern "C" {

int32_t ihtb_mvfit_create(const ihtb_geno* g, const double* Y, int64_t r, const double* z, int64_t q,
                          const ihtb_cfg* cfg, ihtb_mvfit** out) {
    return ihtb_mvfit_create_sharded(g, nullptr, g ? g->p : 0, Y, r, z, q, cfg, out);
}

int32_t ihtb_mvfit_create_sharded(const ihtb_geno* g, ihtb_comm* comm, int64_t p_global, const double* Y, int64_t r,
                                  const double* z, int64_t q, const ihtb_cfg* cfg, ihtb_mvfit** out) {
    return guard([&] {
        IHTB_CHECK(g && Y && z && cfg && out, IHTB_EINVAL, "NULL argument");
        geno_require_ready(g);
        IHTB_CHECK(!geno_is_dense(g), IHTB_EUNSUPPORTED, "multivariate (MvNormal) fits need a PLINK handle: dense matrices "
                                                         "serve univariate fits only");
        IHTB_CHECK(p_global >= g->p, IHTB_EDIM, "p_global is smaller than the local shard");
        IHTB_CHECK(r >= 2 && r <= MV_MAXR, IHTB_EUNSUPPORTED, "multivariate IHT supports 2..20 traits");
        IHTB_CHECK(cfg->sweep_mode == IHTB_SWEEP_FAST || cfg->sweep_mode == IHTB_SWEEP_EXACT ||
                       cfg->sweep_mode == IHTB_SWEEP_PAIR, IHTB_EINVAL, "bad sweep_mode");
        IHTB_CHECK(!cfg->debias, IHTB_EUNSUPPORTED,
                   "Currently the debiasing routine for multivariate IHT is broken, sorry!");   // src/multivariate.jl:570
        IHTB_CHECK(q >= 1, IHTB_EDIM, "z must have at least the intercept row");
        IHTB_CHECK(cfg->k >= 1 && cfg->k <= p_global * r, IHTB_EINVAL, "Multivariate IHT requires 1 <= k <= r*p");
        IHTB_CHECK(cfg->max_iter >= 0 && cfg->max_step >= 0 && cfg->tol > 2.220446049250313e-16, IHTB_EINVAL,
                   "bad max_iter / max_step / tol");
        IHTB_CHECK(g->p * r < (int64_t(1) << 31), IHTB_EDIM, "r*p must be < 2^31");
        IHTB_CUDA(cudaSetDevice(g->device));
        std::unique_ptr<ihtb_mvfit> f(new ihtb_mvfit());
        int64_t n = g->n, p = g->p;
        f->g = g; f->device = g->device; f->n = n; f->p = p; f->q = q; f->r = (int)r; f->cfg = *cfg;
        f->cap = (int)std::max<int64_t>(4096, 4 * cfg->k + 1024);
        f->comm = (comm && comm->nranks > 1) ? comm : nullptr;
        f->j0 = f->comm ? g->j0 : 0;
        f->p_global = f->comm ? p_global : p;
        IHTB_CUDA(cudaStreamCreateWithFlags(&f->s, cudaStreamNonBlocking));
        if (f->comm) {
            // peer-memory areas (collective): n x r products in one all-reduce, candidate blocks in one all-gather
            p2p_setup(f->comm, (size_t)(n * r), 1 + (size_t)f->cap, f->s);
            f->d_xch.alloc(1 + (size_t)f->cap);
            f->d_xchall.alloc((size_t)f->comm->nranks * (1 + (size_t)f->cap));
            f->h_xchall.alloc((size_t)f->comm->nranks * (1 + (size_t)f->cap));
        }
        IHTB_CUDA(cudaEventCreate(&f->ev0)); IHTB_CUDA(cudaEventCreate(&f->ev1));
        f->d_Y.alloc(n * r); f->d_Z.alloc(n * q); f->d_w.alloc(n); f->d_BX.alloc(n * r); f->d_mu.alloc(n * r);
        f->d_resid.alloc(n * r); f->d_R1.alloc(n * r); f->d_V.alloc(n * r); f->d_dfa.alloc(p * r);
        f->d_b0d.alloc(p * r); f->d_mask.alloc(n);
        int nvmax = (int)std::max<int64_t>(2 * r + r * q, r * (r + 1) / 2 + 1);
        f->d_part.alloc((size_t)GLM_MAX_BLOCKS * nvmax); f->d_scal.alloc(nvmax + 8); f->d_C.alloc(r * q);
        size_t cols_cap = 2 * (size_t)f->cap + 64;
        f->d_coef.alloc(cols_cap * r); f->d_gout.alloc(cols_cap * r); f->d_vbar.alloc(r); f->d_sval.alloc(cols_cap);
        f->d_idx.alloc(cols_cap); f->d_cols.alloc(cols_cap); f->d_sidx.alloc(cols_cap); f->d_bounds.alloc(r);
        f->d_keyL.alloc(p * r); f->d_keyU.alloc(p * r); f->d_hist.alloc(2 * 3 * 2048); f->d_sel.alloc(2 + f->cap);
        f->h_scal.alloc(nvmax + 8); f->h_gout.alloc(cols_cap * r); f->h_sel.alloc(2 + f->cap);
        f->sweep_scratch = sweep_scratch_create();
        f->d_b0d.zero(f->s); f->d_hist.zero(f->s);
        IHTB_CUDA(cudaMemcpyAsync(f->d_Y.p, Y, n * r * sizeof(double), cudaMemcpyHostToDevice, f->s));
        IHTB_CUDA(cudaMemcpyAsync(f->d_Z.p, z, n * q * sizeof(double), cudaMemcpyHostToDevice, f->s));
        f->tk = TopkCtx{p * r, f->d_keyL.p, f->d_keyU.p, f->d_hist.p, reinterpret_cast<TopkState*>(f->d_sel.p),
                        f->d_sel.p + 2, f->cap};
        if (f->comm) { f->tk.comm = f->comm; f->tk.p_total = p_global * r; }     // one selection over all shards' entries
        f->sync();
        *out = f.release();
    });
}

int32_t ihtb_mvfit_init(ihtb_mvfit* f, const uint8_t* train_mask) {
    return guard([&] {
        IHTB_CHECK(f, IHTB_EINVAL, "NULL fit handle");
        IHTB_CUDA(cudaSetDevice(f->device));
        f->init(train_mask);
    });
}

int32_t ihtb_mvfit_init_beta(ihtb_mvfit* f, const uint8_t* train_mask) {
    return guard([&] {
        IHTB_CHECK(f, IHTB_EINVAL, "NULL fit handle");
        IHTB_CUDA(cudaSetDevice(f->device));
        f->init(train_mask, /*init_beta=*/true);
    });
}

int32_t ihtb_mvfit_set_k(ihtb_mvfit* f, int64_t k) {
    return guard([&] {
        IHTB_CHECK(f && k >= 1 && 4 * k + 1024 <= f->cap, IHTB_EINVAL, "bad k for this fit handle");
        f->cfg.k = k;
    });
}

int32_t ihtb_mvfit_run(ihtb_mvfit* f, ihtb_result* result, ihtb_iter_trace* trace, int64_t trace_cap) {
    return guard([&] {
        IHTB_CHECK(f, IHTB_EINVAL, "NULL fit handle");
        IHTB_CUDA(cudaSetDevice(f->device));
        f->run(result, trace, trace_cap);
    });
}

int32_t ihtb_mvfit_get(const ihtb_mvfit* f, double* beta, double* c, double* Sigma, double* sigma_g) {
    return guard([&] {
        IHTB_CHECK(f, IHTB_EINVAL, "NULL fit handle");
        const int r = f->r;
        if (beta) {
            std::fill(beta, beta + f->p_global * r, 0.0);
            for (auto& kv : f->bestB) beta[kv.first] = kv.second;          // position j*r + t: r x p column-major
        }
        if (c)      // r x q column-major like Julia's best_C
            for (int t = 0; t < r; ++t)
                for (int64_t l = 0; l < f->q; ++l) c[t + l * r] = f->bestC[t * f->q + l];
        if (Sigma) {  // inv(Gamma) (src/data_structures.jl:274-275)
            std::vector<double> L((size_t)r * r), S((size_t)r * r);
            IHTB_CHECK(chol_lower(r, f->Gamma.data(), L.data()), IHTB_ENUMERIC, "precision matrix is not positive definite");
            spd_inverse(r, L.data(), S.data());
            std::copy(S.begin(), S.end(), Sigma);
        }
        if (sigma_g) std::copy(f->pve.begin(), f->pve.end(), sigma_g);
    });
}

// predict! for mIHTVariable (src/cross_validation.jl:288-299): sum_j,i (Y - mu)^2 w
int32_t ihtb_mvfit_predict(ihtb_mvfit* f, const uint8_t* test_mask, double* mse) {
    return guard([&] {
        IHTB_CHECK(f && mse, IHTB_EINVAL, "NULL argument");
        IHTB_CUDA(cudaSetDevice(f->device));
        f->set_weights(test_mask);
        f->update_xb();
        std::vector<double> G = f->resid_gram();
        double tr = 0.0;
        for (int i = 0; i < f->r; ++i) tr += G[i * f->r + i];
        *mse = tr;
    });
}

int32_t ihtb_mvfit_destroy(ihtb_mvfit* f) {
    return guard([&] {
        if (f) { cudaSetDevice(f->device); delete f; }
    });
}

}  // extern "C"
