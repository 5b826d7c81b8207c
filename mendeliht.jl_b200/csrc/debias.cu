// debias! (reference src/utilities.jl:1014-1020): refit the GLM on the columns of the current support,
//     temp_glm = fit(GeneralizedLinearModel, v.xk, v.y, v.d, v.l);  b[idx] = temp_glm.pp.beta0
// i.e. GLM.jl's IRLS with default arguments on xk = x[:, idx] (ALL n samples, no covariates, no intercept).  GLM.jl is
// not vendored in the reference tree; its `_fit!` loop is restated here (oracle twin: oracle/glm.py::glm_fit):
//   eta = linkfun(mustart(y)); beta = WLS(wrkresid + eta); then Newton steps delta = (X'WX)^-1 X'W wrkresid with
//   step-halving while dev > devold + rtol*dev; stop when devold - dev < max(rtol*devold, atol); 30 iterations at most.
// Device work per IRLS evaluation: one pass over the decoded n x k block (eta, mu, working weight/residual, deviance)
// and one tiled weighted Gram kernel [X u]' W [X u]; the k x k Cholesky solve runs on the host.  All reductions have a
// fixed order (deterministic).
#include "debias.cuh"
#include "comm.cuh"
#include "glm.cuh"

namespace ihtb {

constexpr int DB_TILE = 16;          // columns per Gram tile
constexpr int DB_ROWS = 128;         // samples staged per step
constexpr int DB_MAX_CHUNKS = 64;    // sample chunks (partial Gram sums) per tile pair

__device__ __forceinline__ double db_linkfun(int link, double mu) {
    switch (link) {
        case IHTB_LINK_IDENTITY: return mu;
        case IHTB_LINK_LOGIT: return log(mu / (1.0 - mu));
        case IHTB_LINK_LOG: return log(mu);
        case IHTB_LINK_PROBIT: return normcdfinv(mu);
        case IHTB_LINK_CLOGLOG: return log(-log1p(-mu));
        case IHTB_LINK_CAUCHIT: return tan(3.141592653589793 * (mu - 0.5));
        case IHTB_LINK_SQRT: return sqrt(mu);
        case IHTB_LINK_INVERSE: return 1.0 / mu;
        case IHTB_LINK_INVSQ: return 1.0 / (mu * mu);
    }
    return NAN;
}

__device__ __forceinline__ double db_mustart(int dist, double y) {   // GLM.jl mustart(d, y, wt = 1)
    switch (dist) {
        case IHTB_NORMAL: return y;
        case IHTB_BERNOULLI: return (y + 0.5) / 2.0;
        case IHTB_POISSON: return y + 0.1;
        case IHTB_NEGBIN: return y == 0.0 ? y + 1.0 / 6.0 : y;
    }
    return NAN;
}

// xk[c*n + i] = x[i, cols[c]] through the getindex formula (same arithmetic as k_decode)
__global__ void k_decode_cols(GenoView gv, int center, const int64_t* __restrict__ cols, int64_t k,
                              double* __restrict__ out) {
    const int64_t n = gv.n;
    int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n * k) return;
    const int64_t c = t / n, i = t % n, j = cols[c];
    if (j < 0) { out[t] = 0.0; return; }          // column of another shard: filled in by the all-reduce
    uint32_t code = (*gv_ptr(gv, j, i >> 2) >> (2 * (i & 3))) & 3u;
    double m = gv.mu[j];
    double g = (code == 2) ? 1.0 : (code == 3) ? 2.0 : (code == 1) ? (gv.impute ? m : 0.0) : 0.0;
    if (center) g = __dsub_rn(g, m);
    out[t] = __dmul_rn(g, gv.sinv[j]);
}

// One IRLS evaluation.  init = 1: eta = linkfun(mustart(y)) and u = wrkresid + eta (the working response);
// init = 0: eta = xk * beta and u = wrkresid.  Writes w (working weights), u (column k of xk), block deviance sums.
__global__ void __launch_bounds__(256)
k_irls_eval(int64_t n, int k, double* __restrict__ xk, const double* __restrict__ beta, const double* __restrict__ y,
            int dist, int link, double nb_r, int init, double* __restrict__ w, double* __restrict__ part) {
    __shared__ double sh[32];
    __shared__ double sb[DB_MAX_K];
    for (int c = threadIdx.x; c < k; c += blockDim.x) sb[c] = init ? 0.0 : beta[c];
    __syncthreads();
    double dev = 0.0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double yi = y[i];
        double eta;
        if (init) {
            eta = db_linkfun(link, db_mustart(dist, yi));
        } else {
            eta = 0.0;
            for (int c = 0; c < k; ++c) eta = fma(xk[(int64_t)c * n + i], sb[c], eta);
        }
        const double mu = glm_linkinv(link, eta);
        const double dmu = glm_mueta(link, eta);
        const double wrkres = (yi - mu) / dmu;
        w[i] = dmu * dmu / glm_var(dist, mu, nb_r);
        xk[(int64_t)k * n + i] = init ? wrkres + eta : wrkres;
        dev += glm_devresid(dist, yi, mu, nb_r);
    }
    dev = block_sum(dev, sh);
    if (threadIdx.x == 0) part[blockIdx.x] = dev;
}

__global__ void k_sum_in_order(const double* __restrict__ part, int nparts, double* __restrict__ out) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        double a = 0.0;
        for (int t = 0; t < nparts; ++t) a += part[t];
        *out = a;
    }
}

// Weighted Gram of the kk = k + 1 columns of xk: G[a][b] = sum_i w_i xk[a][i] xk[b][i] for tile pairs ta <= tb.
// grid = (n_tile_pairs, n_chunks); thread (la, lb) of the 16 x 16 tile accumulates its entry over the chunk's samples
// staged through shared memory; partial sums go to part[chunk][pair][256].
__global__ void __launch_bounds__(DB_TILE * DB_TILE)
k_gram(int64_t n, int kk, const double* __restrict__ xk, const double* __restrict__ w, int ntiles, int64_t chunk_rows,
       double* __restrict__ part) {
    __shared__ double sa[DB_TILE][DB_ROWS + 1];
    __shared__ double sbt[DB_TILE][DB_ROWS + 1];
    __shared__ double sw[DB_ROWS];
    // decode the linear pair index into (ta, tb), ta <= tb
    int pair = blockIdx.x, ta = 0;
    while (pair >= ntiles - ta) { pair -= ntiles - ta; ++ta; }
    const int tb = ta + pair;
    const int la = threadIdx.x / DB_TILE, lb = threadIdx.x % DB_TILE;
    const int64_t i_beg = blockIdx.y * chunk_rows;
    const int64_t i_end = (i_beg + chunk_rows < n) ? i_beg + chunk_rows : n;
    double acc = 0.0;
    for (int64_t i0 = i_beg; i0 < i_end; i0 += DB_ROWS) {
        const int rows = (int)((i_end - i0 < DB_ROWS) ? (i_end - i0) : DB_ROWS);
        __syncthreads();
        for (int e = threadIdx.x; e < DB_TILE * DB_ROWS; e += blockDim.x) {
            const int c = e / DB_ROWS, r = e % DB_ROWS;
            const int ca = ta * DB_TILE + c, cb = tb * DB_TILE + c;
            sa[c][r] = (r < rows && ca < kk) ? xk[(int64_t)ca * n + i0 + r] : 0.0;
            sbt[c][r] = (r < rows && cb < kk) ? xk[(int64_t)cb * n + i0 + r] : 0.0;
        }
        for (int r = threadIdx.x; r < DB_ROWS; r += blockDim.x) sw[r] = (r < rows) ? w[i0 + r] : 0.0;
        __syncthreads();
#pragma unroll 8
        for (int r = 0; r < DB_ROWS; ++r) acc = fma(sw[r] * sa[la][r], sbt[lb][r], acc);
    }
    part[((int64_t)blockIdx.y * gridDim.x + blockIdx.x) * (DB_TILE * DB_TILE) + threadIdx.x] = acc;
}

// G[a*kk + b] (full symmetric kk x kk) = sum over chunks, in chunk order
__global__ void k_gram_fin(int kk, int ntiles, int npairs, int nchunks, const double* __restrict__ part,
                           double* __restrict__ G) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= npairs * DB_TILE * DB_TILE) return;
    int pair = t / (DB_TILE * DB_TILE), l = t % (DB_TILE * DB_TILE);
    int pr = pair, ta = 0;
    while (pr >= ntiles - ta) { pr -= ntiles - ta; ++ta; }
    const int tb = ta + pr;
    const int a = ta * DB_TILE + l / DB_TILE, b = tb * DB_TILE + l % DB_TILE;
    if (a >= kk || b >= kk) return;
    double s = 0.0;
    for (int c = 0; c < nchunks; ++c) s += part[((int64_t)c * npairs + pair) * (DB_TILE * DB_TILE) + l];
    G[a * kk + b] = s;
    G[b * kk + a] = s;
}

// in-place Cholesky solve of the k x k system A x = rhs (A symmetric, row-major, leading dimension ld)
static bool chol_solve(std::vector<double>& A, int k, std::vector<double>& x) {
    for (int j = 0; j < k; ++j) {
        double d = A[j * k + j];
        for (int t = 0; t < j; ++t) d -= A[j * k + t] * A[j * k + t];
        if (!(d > 0.0)) return false;
        d = std::sqrt(d);
        A[j * k + j] = d;
        for (int i = j + 1; i < k; ++i) {
            double v = A[i * k + j];
            for (int t = 0; t < j; ++t) v -= A[i * k + t] * A[j * k + t];
            A[i * k + j] = v / d;
        }
    }
    for (int i = 0; i < k; ++i) {           // L z = rhs
        double v = x[i];
        for (int t = 0; t < i; ++t) v -= A[i * k + t] * x[t];
        x[i] = v / A[i * k + i];
    }
    for (int i = k - 1; i >= 0; --i) {      // L' x = z
        double v = x[i];
        for (int t = i + 1; t < k; ++t) v -= A[t * k + i] * x[t];
        x[i] = v / A[i * k + i];
    }
    return true;
}

void DebiasWs::ensure(int64_t n, int k) {
    const int kk = k + 1;
    if (xk.n < (size_t)(n * kk)) xk.alloc((size_t)(n * kk));
    if (w.n < (size_t)n) w.alloc((size_t)n);
    const int ntiles = (kk + DB_TILE - 1) / DB_TILE;
    const int npairs = ntiles * (ntiles + 1) / 2;
    if (gpart.n < (size_t)DB_MAX_CHUNKS * npairs * DB_TILE * DB_TILE) gpart.alloc((size_t)DB_MAX_CHUNKS * npairs * DB_TILE * DB_TILE);
    if (G.n < (size_t)(kk * kk + 1)) { G.alloc((size_t)(kk * kk + 1)); hG.alloc((size_t)(kk * kk + 1)); }
    if (dpart.n < 1024) dpart.alloc(1024);
    if (beta.n < (size_t)DB_MAX_K) { beta.alloc(DB_MAX_K); hbeta.alloc(DB_MAX_K); }
}

void debias_irls(const ihtb_geno* g, const double* d_y, int dist, int link, double nb_r, const int64_t* d_cols, int k,
                 double* beta_out, DebiasWs& ws, cudaStream_t s, ihtb_comm* comm) {
    IHTB_CHECK(k >= 1 && k <= DB_MAX_K, IHTB_EUNSUPPORTED,
               "debiasing supports at most " + std::to_string(DB_MAX_K) + " predictors in the support");
    const int64_t n = g->n;
    const int kk = k + 1;
    ws.ensure(n, k);
    if (geno_is_dense(g)) dense_decode_cols(g, d_cols, k, ws.xk.p, s);
    else IHTB_LAUNCH(k_decode_cols, (unsigned)ceil_div(n * k, 256), 256, 0, s, geno_view(g), g->center, d_cols, (int64_t)k, ws.xk.p);
    // SNP-sharded fits: every rank decodes its own support columns (zeros elsewhere); one all-reduce of the n x k block
    // gives all ranks the same dense matrix, and the refit then runs replicated
    if (comm) comm_allreduce_sum_f64(comm, ws.xk.p, (size_t)(n * k), s);
    const int eval_grid = (int)std::min<int64_t>(1024, ceil_div(n, 256));
    const int ntiles = (kk + DB_TILE - 1) / DB_TILE;
    const int npairs = ntiles * (ntiles + 1) / 2;
    int nchunks = (int)std::min<int64_t>(DB_MAX_CHUNKS, ceil_div(n, 8 * DB_ROWS));
    if (nchunks < 1) nchunks = 1;
    const int64_t chunk_rows = ceil_div(ceil_div(n, nchunks), DB_ROWS) * DB_ROWS;
    nchunks = (int)ceil_div(n, chunk_rows);

    // evaluate at `b` (NULL: the mustart initialisation), return the deviance; w / u stay on the device
    auto eval = [&](const double* b) -> double {
        if (b) {
            memcpy(ws.hbeta.p, b, (size_t)k * sizeof(double));
            IHTB_CUDA(cudaMemcpyAsync(ws.beta.p, ws.hbeta.p, (size_t)k * sizeof(double), cudaMemcpyHostToDevice, s));
        }
        IHTB_LAUNCH(k_irls_eval, eval_grid, 256, 0, s, n, k, ws.xk.p, ws.beta.p, d_y, dist, link, nb_r, b ? 0 : 1, ws.w.p,
                    ws.dpart.p);
        IHTB_LAUNCH(k_sum_in_order, 1, 32, 0, s, ws.dpart.p, eval_grid, ws.G.p + kk * kk);
        IHTB_CUDA(cudaMemcpyAsync(ws.hG.p + kk * kk, ws.G.p + kk * kk, sizeof(double), cudaMemcpyDeviceToHost, s));
        IHTB_CUDA(cudaStreamSynchronize(s));
        double dev = ws.hG.p[kk * kk];
        return std::isnan(dev) ? INFINITY : dev;
    };
    // delta = (X'WX)^-1 X'W u for the current w / u
    auto delbeta = [&](std::vector<double>& delta) {
        IHTB_LAUNCH(k_gram, dim3(npairs, nchunks), DB_TILE * DB_TILE, 0, s, n, kk, ws.xk.p, ws.w.p, ntiles, chunk_rows, ws.gpart.p);
        IHTB_LAUNCH(k_gram_fin, (unsigned)ceil_div(npairs * DB_TILE * DB_TILE, 256), 256, 0, s, kk, ntiles, npairs, nchunks,
                    ws.gpart.p, ws.G.p);
        IHTB_CUDA(cudaMemcpyAsync(ws.hG.p, ws.G.p, (size_t)kk * kk * sizeof(double), cudaMemcpyDeviceToHost, s));
        IHTB_CUDA(cudaStreamSynchronize(s));
        std::vector<double> A((size_t)k * k);
        delta.assign((size_t)k, 0.0);
        for (int a = 0; a < k; ++a) {
            for (int b = 0; b < k; ++b) A[(size_t)a * k + b] = ws.hG.p[a * kk + b];
            delta[a] = ws.hG.p[a * kk + k];
        }
        IHTB_CHECK(chol_solve(A, k, delta), IHTB_ENUMERIC,
                   "debias: X'WX of the support is not positive definite (PosDefException in the reference)");
    };

    const double rtol = 1e-6, atol = 1e-6, minstepfac = 0.001;
    const int maxiter = 30;
    std::vector<double> beta0, delta, trial((size_t)k);
    eval(nullptr);
    delbeta(beta0);
    double devold = eval(beta0.data());
    for (int it = 0; it < maxiter; ++it) {
        double f = 1.0;
        delbeta(delta);
        for (int c = 0; c < k; ++c) trial[c] = beta0[c] + delta[c];
        double dev = eval(trial.data());
        while (dev > devold + rtol * dev) {
            f /= 2.0;
            IHTB_CHECK(f > minstepfac, IHTB_ENUMERIC, "debias: step-halving failed");
            for (int c = 0; c < k; ++c) trial[c] = beta0[c] + f * delta[c];
            dev = eval(trial.data());
        }
        for (int c = 0; c < k; ++c) beta0[c] += f * delta[c];
        if (devold - dev < std::max(rtol * devold, atol)) {
            for (int c = 0; c < k; ++c) beta_out[c] = beta0[c];
            return;
        }
        devold = dev;
    }
    throw Error(IHTB_ENUMERIC, "debias: failure to converge after 30 iterations.");
}

}  // namespace ihtb
