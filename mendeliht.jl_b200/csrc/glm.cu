// Fused elementwise GLM kernels + deterministic reductions over the n-vectors of one fit.
// Replace update_mu! (reference src/utilities.jl:74-82), the clamp and z*c of update_xb! (:113-117),
// deviance / loglikelihood (:9-61), the residual loop of score! (:128-134, incl. df2 = Z'r) and the
// sqrt(W) weighting + dot of iht_stepsize! (:744-756).  Link / variance / deviance / logpdf formulas are those
// of GLM.jl 1.x and Distributions.jl 0.25 (SURVEY.md App. B).
#include "glm.cuh"

namespace ihtb {

constexpr int GLM_THREADS = 256;

static inline int glm_grid(int64_t n) {
    int64_t b = ceil_div(n, GLM_THREADS);
    return (int)(b < 1 ? 1 : (b > GLM_MAX_BLOCKS ? GLM_MAX_BLOCKS : b));
}

// In-kernel finalisation: every CTA calls this after thread 0 wrote the CTA's nv partial sums to part[blockIdx.x * nv ..].
// The CTA that arrives last (ticket counter `done`, reset for the next launch) reduces all of them exactly like k_finalize:
// one warp per value, lanes stride over the CTAs, fixed shuffle tree -- bit-identical sums, one launch less.
__device__ __forceinline__ void cta_finalize(const double* part, int nv, double* out, unsigned* done,
                                             double* mean_out = nullptr, int64_t n = 1) {
    __shared__ int s_last;
    if (threadIdx.x == 0) {
        __threadfence();                                   // this CTA's partial sums before its ticket
        const unsigned t = atomicAdd(done, 1u);
        s_last = (t == gridDim.x - 1);
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();                                       // the other CTAs' sums after the last ticket
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const int nblocks = (int)gridDim.x;
    for (int v = warp; v < nv; v += nw) {
        double a = 0.0;
        for (int b = lane; b < nblocks; b += 32) a += __ldcg(part + (int64_t)b * nv + v);
        a = warp_sum(a);
        if (lane == 0) {
            out[v] = a;
            if (mean_out && v == 0) mean_out[0] = a / (double)n;
        }
    }
    if (threadIdx.x == 0) *done = 0u;
}

// xb (clamped in place unless Normal), zc = Z c (clamped), mu = linkinv(xb + zc) [or linkinv(xb) when !add_zc],
// partial sums: [0] sum w*devresid, [1] sum w*logpdf (phi-free part; unused for Normal), [2] sum w
__global__ void __launch_bounds__(GLM_THREADS)
k_glm_mu(int64_t n, int64_t q, const double* __restrict__ Z, const double* __restrict__ c, double* __restrict__ xb,
         double* __restrict__ zc, double* __restrict__ mu, const double* __restrict__ y, const double* __restrict__ w,
         int dist, int link, double nb_r, int add_zc, double* __restrict__ part, double* __restrict__ out = nullptr,
         unsigned* __restrict__ done = nullptr) {
    __shared__ double sh[32];
    // blockIdx.y = model of a batched evaluation (glm_mu_batched): every model has its own c, xb, zc, mu and partial
    // sums, laid out back to back, and is reduced exactly like a single model (same blocks, same order)
    c += blockIdx.y * q; xb += blockIdx.y * n; zc += blockIdx.y * n; mu += blockIdx.y * n;
    part += (int64_t)blockIdx.y * gridDim.x * 3;
    double a_dev = 0.0, a_lp = 0.0, a_w = 0.0;
    const bool clampit = dist != IHTB_NORMAL;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double z = 0.0;
        for (int64_t l = 0; l < q; ++l) z += Z[i + l * n] * c[l];
        double x = xb[i];
        if (clampit) {
            x = fmin(fmax(x, -20.0), 20.0);
            z = fmin(fmax(z, -20.0), 20.0);
            xb[i] = x;
        }
        zc[i] = z;
        double m = glm_linkinv(link, add_zc ? x + z : x);
        mu[i] = m;
        double wi = w[i], yi = y[i];
        a_dev += wi * glm_devresid(dist, yi, m, nb_r);
        if (dist != IHTB_NORMAL) a_lp += wi * glm_logpdf_nophi(dist, yi, m, nb_r);
        a_w += wi;
    }
    a_dev = block_sum(a_dev, sh);
    a_lp = block_sum(a_lp, sh);
    a_w = block_sum(a_w, sh);
    if (threadIdx.x == 0) {
        part[blockIdx.x * 3 + 0] = a_dev;
        part[blockIdx.x * 3 + 1] = a_lp;
        part[blockIdx.x * 3 + 2] = a_w;
    }
    if (done) cta_finalize(part, 3, out + blockIdx.y * 3, done + blockIdx.y);
}

// r_i = mueta(eta_i)/glmvar(mu_i) * (y_i - mu_i) * w_i ; partials [0] sum r, [1] sum |r|, [2..2+q) Z'r
__global__ void __launch_bounds__(GLM_THREADS)
k_score(int64_t n, int64_t q, const double* __restrict__ Z, const double* __restrict__ xb,
        const double* __restrict__ zc, const double* __restrict__ mu, const double* __restrict__ y,
        const double* __restrict__ w, int dist, int link, double nb_r, double* __restrict__ r,
        double* __restrict__ part, double* __restrict__ out = nullptr, unsigned* __restrict__ done = nullptr,
        double* __restrict__ mean_out = nullptr) {
    __shared__ double sh[32];
    const int nv = 2 + (int)q;
    double a_r = 0.0, a_abs = 0.0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double eta = xb[i] + zc[i];
        double m = mu[i];
        double ri = glm_mueta(link, eta) / glm_var(dist, m, nb_r) * (y[i] - m) * w[i];
        r[i] = ri;
        a_r += ri;
        a_abs += fabs(ri);
    }
    a_r = block_sum(a_r, sh);
    a_abs = block_sum(a_abs, sh);
    if (threadIdx.x == 0) {
        part[blockIdx.x * nv + 0] = a_r;
        part[blockIdx.x * nv + 1] = a_abs;
    }
    // df2 = Z'r (second pass over this block's rows; r was just written by the same threads)
    for (int64_t l = 0; l < q; ++l) {
        double a = 0.0;
        for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
            a += Z[i + l * n] * r[i];
        a = block_sum(a, sh);
        if (threadIdx.x == 0) part[blockIdx.x * nv + 2 + l] = a;
    }
    if (done) cta_finalize(part, nv, out, done, mean_out, n);
}

// xgk_i = (xs_i + sum_l Z[i,l] d2_l) * sqrt(mueta^2 / glmvar) * w_i ; partial [0] = sum xgk_i^2
__global__ void __launch_bounds__(GLM_THREADS)
k_stepsize(int64_t n, int64_t q, const double* __restrict__ Z, const double* __restrict__ d2,
           const double* __restrict__ d2mask, const double* __restrict__ xs, const double* __restrict__ xb,
           const double* __restrict__ zc,
           const double* __restrict__ mu, const double* __restrict__ w, int dist, int link, double nb_r,
           double* __restrict__ part, double* __restrict__ out = nullptr, unsigned* __restrict__ done = nullptr) {
    __shared__ double sh[32];
    double a = 0.0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double zd = 0.0;
        for (int64_t l = 0; l < q; ++l) zd += Z[i + l * n] * (d2mask ? d2[l] * d2mask[l] : d2[l]);
        double g = glm_mueta(link, xb[i] + zc[i]);
        double sw = sqrt(g * g / glm_var(dist, mu[i], nb_r)) * w[i];
        double v = (xs[i] + zd) * sw;
        a += v * v;
    }
    a = block_sum(a, sh);
    if (threadIdx.x == 0) part[blockIdx.x] = a;
    if (done) cta_finalize(part, 1, out, done);
}

// partials [0] sum a_i, [1] sum b_i   (means for pve)
__global__ void __launch_bounds__(GLM_THREADS)
k_sum2(int64_t n, const double* __restrict__ a, const double* __restrict__ b, double* __restrict__ part) {
    __shared__ double sh[32];
    double sa = 0.0, sb = 0.0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        sa += a[i]; sb += b[i];
    }
    sa = block_sum(sa, sh); sb = block_sum(sb, sh);
    if (threadIdx.x == 0) { part[blockIdx.x * 2] = sa; part[blockIdx.x * 2 + 1] = sb; }
}
// partials [0] sum (a_i - ma)^2, [1] sum (b_i - mb)^2
__global__ void __launch_bounds__(GLM_THREADS)
k_ssq2(int64_t n, const double* __restrict__ a, double ma, const double* __restrict__ b, double mb,
       double* __restrict__ part) {
    __shared__ double sh[32];
    double sa = 0.0, sb = 0.0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double da = a[i] - ma, db = b[i] - mb;
        sa += da * da; sb += db * db;
    }
    sa = block_sum(sa, sh); sb = block_sum(sb, sh);
    if (threadIdx.x == 0) { part[blockIdx.x * 2] = sa; part[blockIdx.x * 2 + 1] = sb; }
}

// w_i = mask_i ? 1 : 0 ; partials [0] sum w, [1] sum y*w
__global__ void __launch_bounds__(GLM_THREADS)
k_set_weights(int64_t n, const uint8_t* __restrict__ mask, const double* __restrict__ y, double* __restrict__ w,
              double* __restrict__ part) {
    __shared__ double sh[32];
    double sw = 0.0, sy = 0.0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double wi = (mask == nullptr || mask[i]) ? 1.0 : 0.0;
        w[i] = wi;
        sw += wi;
        sy += y[i] * wi;
    }
    sw = block_sum(sw, sh); sy = block_sum(sy, sh);
    if (threadIdx.x == 0) { part[blockIdx.x * 2] = sw; part[blockIdx.x * 2 + 1] = sy; }
}

// out[v] = sum_b part[b*nv + v]: one warp per value, lanes stride over the blocks, fixed shuffle tree (deterministic)
// mean_out (optional): also writes out[0] / n, the mean the sweep centres the residual with (saves a launch)
__global__ void k_finalize(const double* __restrict__ part, int nblocks, int nv, double* __restrict__ out,
                           double* __restrict__ mean_out = nullptr, int64_t n = 1) {
    part += (int64_t)blockIdx.y * nblocks * nv; out += blockIdx.y * nv;       // batched: one row of sums per model
    int v = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (v >= nv) return;
    double a = 0.0;
    for (int b = lane; b < nblocks; b += 32) a += part[b * nv + v];
    a = warp_sum(a);
    if (lane == 0) {
        out[v] = a;
        if (mean_out && v == 0 && blockIdx.y == 0) mean_out[0] = a / (double)n;
    }
}

__global__ void k_mean_from_sum(const double* __restrict__ scal, int64_t n, double* __restrict__ out) {
    out[0] = scal[0] / (double)n;
}

// ---- init_beta helpers (reference initialize_beta! / linreg!, src/utilities.jl:776-842) ------------------------------
__global__ void k_wy(int64_t n, const double* __restrict__ w, const double* __restrict__ y, double* __restrict__ out) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) out[i] = w[i] * y[i];
}
// regression of y on [1, x_j] from N = sum w, SY = sum w y, sx, sxx, sxy by a 2x2 Cholesky; a failed factorisation
// leaves (SY, sxy) like the reference's try/catch (src/utilities.jl:776-842); the slope is clamped to [-2, 2]
__device__ __forceinline__ void init_beta_regress(double N, double SY, double sx, double sxx, double sxy, double& beta,
                                                  double& icpt) {
    double slope = sxy;
    icpt = SY;
    const double u11 = sqrt(N), u12 = sx / u11, dd = sxx - u12 * u12;
    if (N > 0.0 && dd > 0.0) {
        const double u22 = sqrt(dd), t1 = SY / u11, t2 = (sxy - u12 * t1) / u22;
        slope = t2 / u22;
        icpt = (t1 - u12 * slope) / u11;
    }
    beta = fmin(fmax(slope, -2.0), 2.0);
}
// per SNP: regression of y on [1, x_j] over the weighted samples from the class sums.  part[block] = sum of intercepts.
__global__ void __launch_bounds__(GLM_THREADS)
k_init_beta(int64_t p, const double* __restrict__ W1, const double* __restrict__ W2, const double* __restrict__ Wm,
            const double* __restrict__ Y1, const double* __restrict__ Y2, const double* __restrict__ Ym, double N,
            double SY, const double* __restrict__ mu, const double* __restrict__ sinv, int impute,
            double* __restrict__ beta, double* __restrict__ part) {
    __shared__ double sh[32];
    double acc = 0.0;
    for (int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j < p; j += (int64_t)gridDim.x * blockDim.x) {
        const double m = mu[j], si = sinv[j];
        const double a0 = (0.0 - m) * si, a1 = (1.0 - m) * si, a2 = (2.0 - m) * si, am = impute ? 0.0 : a0;
        const double w1 = W1[j], w2 = W2[j], wm = Wm[j], w0 = N - w1 - w2 - wm;
        const double y1 = Y1[j], y2 = Y2[j], ym = Ym[j], y0 = SY - y1 - y2 - ym;
        const double sx = a0 * w0 + a1 * w1 + a2 * w2 + am * wm;
        const double sxx = a0 * a0 * w0 + a1 * a1 * w1 + a2 * a2 * w2 + am * am * wm;
        const double sxy = a0 * y0 + a1 * y1 + a2 * y2 + am * ym;
        double icpt;
        init_beta_regress(N, SY, sx, sxx, sxy, beta[j], icpt);
        acc += icpt;
    }
    acc = block_sum(acc, sh);
    if (threadIdx.x == 0) part[blockIdx.x] = acc;
}
// the same regressions from per-column moments (dense handles: sum w x, sum w x^2, sum w y x, dense.cu)
__global__ void __launch_bounds__(GLM_THREADS)
k_init_beta_moments(int64_t p, const double* __restrict__ SX, const double* __restrict__ SXX,
                    const double* __restrict__ SXY, double N, double SY, double* __restrict__ beta,
                    double* __restrict__ part) {
    __shared__ double sh[32];
    double acc = 0.0;
    for (int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j < p; j += (int64_t)gridDim.x * blockDim.x) {
        double icpt;
        init_beta_regress(N, SY, SX[j], SXX[j], SXY[j], beta[j], icpt);
        acc += icpt;
    }
    acc = block_sum(acc, sh);
    if (threadIdx.x == 0) part[blockIdx.x] = acc;
}
// covariates l = 1..q-1: partial sums [3(l-1)+0] sum w z, [+1] sum w z^2, [+2] sum w z y
__global__ void __launch_bounds__(GLM_THREADS)
k_cov_sums(int64_t n, int64_t q, const double* __restrict__ Z, const double* __restrict__ y,
           const double* __restrict__ w, double* __restrict__ part) {
    __shared__ double sh[32];
    const int nv = 3 * ((int)q - 1);
    for (int64_t l = 1; l < q; ++l) {
        double a = 0.0, b = 0.0, c = 0.0;
        for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
            double z = Z[i + l * n], wi = w[i];
            a += wi * z; b += wi * z * z; c += wi * z * y[i];
        }
        a = block_sum(a, sh); b = block_sum(b, sh); c = block_sum(c, sh);
        if (threadIdx.x == 0) {
            part[blockIdx.x * nv + 3 * (l - 1)] = a;
            part[blockIdx.x * nv + 3 * (l - 1) + 1] = b;
            part[blockIdx.x * nv + 3 * (l - 1) + 2] = c;
        }
    }
}

// ---- launchers ------------------------------------------------------------------------------------
void init_beta_products(GlmCtx& c, double* d_wy, cudaStream_t s) {
    IHTB_LAUNCH(k_wy, (unsigned)ceil_div(c.n, 256), 256, 0, s, c.n, c.w, c.y, d_wy);
}
void init_beta_solve(GlmCtx& c, int64_t p, const double* W1, const double* W2, const double* Wm, const double* Y1,
                     const double* Y2, const double* Ym, double N, double SY, const double* mu, const double* sinv,
                     int impute, double* d_beta, cudaStream_t s) {
    int grid = glm_grid(p);
    IHTB_LAUNCH(k_init_beta, grid, GLM_THREADS, 0, s, p, W1, W2, Wm, Y1, Y2, Ym, N, SY, mu, sinv, impute, d_beta, c.part);
    IHTB_LAUNCH(k_finalize, 1, 32, 0, s, c.part, grid, 1, c.scal);
}
void init_beta_solve_moments(GlmCtx& c, int64_t p, const double* SX, const double* SXX, const double* SXY, double N,
                             double SY, double* d_beta, cudaStream_t s) {
    int grid = glm_grid(p);
    IHTB_LAUNCH(k_init_beta_moments, grid, GLM_THREADS, 0, s, p, SX, SXX, SXY, N, SY, d_beta, c.part);
    IHTB_LAUNCH(k_finalize, 1, 32, 0, s, c.part, grid, 1, c.scal);
}
void init_beta_cov_sums(GlmCtx& c, cudaStream_t s) {
    int grid = glm_grid(c.n);
    int nv = 3 * ((int)c.q - 1);
    IHTB_LAUNCH(k_cov_sums, grid, GLM_THREADS, 0, s, c.n, c.q, c.Z, c.y, c.w, c.part);
    IHTB_LAUNCH(k_finalize, (unsigned)ceil_div(nv, 4), 128, 0, s, c.part, grid, nv, c.scal);
}
void glm_mean_from_sum(GlmCtx& c, double* d_mean, cudaStream_t s) {
    IHTB_LAUNCH(k_mean_from_sum, 1, 1, 0, s, c.scal, c.n, d_mean);
}
void glm_mu(GlmCtx& c, const double* d_c, int add_zc, cudaStream_t s) {
    int grid = glm_grid(c.n);
    IHTB_LAUNCH(k_glm_mu, grid, GLM_THREADS, 0, s, c.n, c.q, c.Z, d_c, c.xb, c.zc, c.mu, c.y, c.w, c.dist, c.link,
                c.nb_r, add_zc, c.part, c.scal, c.done);
    if (!c.done) IHTB_LAUNCH(k_finalize, 1, 96, 0, s, c.part, grid, 3, c.scal);
}
// M models at once (the gradient step and its backtracks): xbM / zcM / muM are n x M, d_cM is q x M, d_scalM gets
// [dev, lp, sum w] per model.  Per model the arithmetic is that of glm_mu.
void glm_mu_batched(GlmCtx& c, const double* d_cM, int M, double* xbM, double* zcM, double* muM, double* d_partM,
                    double* d_scalM, cudaStream_t s) {
    int grid = glm_grid(c.n);
    IHTB_LAUNCH(k_glm_mu, dim3(grid, M), GLM_THREADS, 0, s, c.n, c.q, c.Z, d_cM, xbM, zcM, muM, c.y, c.w, c.dist, c.link,
                c.nb_r, 1, d_partM, d_scalM, c.done);
    if (!c.done) IHTB_LAUNCH(k_finalize, dim3(1, M), 96, 0, s, d_partM, grid, 3, d_scalM);
}
// ---- the gradient step and its backtracks decided on the device (fit.cu one_step_fused) ------------------------------
// scalM[3m..] = deviance, sum of log-densities, sum of weights of candidate model m (eta / 2^m).  pick[1 + m] = its
// loglikelihood (src/utilities.jl:9-20: Normal uses phi = deviance / length(y)), pick[0] = the model the reference's
// loop `while prev_logl > logl && step < max_step` (src/utilities.jl:484-486) ends at.
__global__ void k_pick_model(const double* __restrict__ scalM, int M, double old_logl, int max_step, int dist, int64_t n,
                             double* __restrict__ pick) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    for (int m = 0; m < M; ++m) {
        const double dev = scalM[3 * m], lp = scalM[3 * m + 1], sw = scalM[3 * m + 2];
        double l = lp;
        if (dist == IHTB_NORMAL) {
            const double phi = dev / (double)n, sigma = sqrt(phi);
            l = -0.5 * (dev / phi) - sw * (0.5 * log(2.0 * 3.14159265358979323846) + log(sigma));
        }
        pick[1 + m] = l;
    }
    int w = 0;
    while (old_logl > pick[1 + w] && w < max_step) ++w;
    pick[0] = (double)w;
}
__global__ void k_take_model(const double* __restrict__ pick, int64_t n, const double* __restrict__ xbM,
                             const double* __restrict__ zcM, const double* __restrict__ muM, double* __restrict__ xb,
                             double* __restrict__ zc, double* __restrict__ mu) {
    const int64_t off = (int64_t)pick[0] * n;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        xb[i] = xbM[off + i]; zc[i] = zcM[off + i]; mu[i] = muM[off + i];
    }
}
// coefficients of the step-size product X[:, supp] df[supp] for the WINNER's support (a subset of the union the
// exact gradient was gathered for), and its covariate mask
__global__ void k_winner_coef(const double* __restrict__ pick, const double* __restrict__ coefM, int64_t U,
                              const double* __restrict__ df_uni, double* __restrict__ coef_out,
                              const double* __restrict__ cM, int64_t q, double* __restrict__ mask_out) {
    const int64_t w = (int64_t)pick[0];
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t < U) coef_out[t] = coefM[t + w * U] != 0.0 ? df_uni[t] : 0.0;
    if (t < q) mask_out[t] = cM[t + w * q] != 0.0 ? 1.0 : 0.0;
}
void glm_pick_model(GlmCtx& c, const double* d_scalM, int M, double old_logl, int max_step, double* d_pick,
                    const double* xbM, const double* zcM, const double* muM, cudaStream_t s) {
    IHTB_LAUNCH(k_pick_model, 1, 32, 0, s, d_scalM, M, old_logl, max_step, c.dist, c.n, d_pick);
    IHTB_LAUNCH(k_take_model, glm_grid(c.n), GLM_THREADS, 0, s, d_pick, c.n, xbM, zcM, muM, c.xb, c.zc, c.mu);
}
void glm_winner_coef(const double* d_pick, const double* d_coefM, int64_t U, const double* d_df_uni, double* d_coef_out,
                     const double* d_cM, int64_t q, double* d_mask_out, cudaStream_t s) {
    const int64_t m = U > q ? U : q;
    IHTB_LAUNCH(k_winner_coef, (unsigned)ceil_div(m > 0 ? m : 1, 128), 128, 0, s, d_pick, d_coefM, U, d_df_uni, d_coef_out,
                d_cM, q, d_mask_out);
}

void glm_score(GlmCtx& c, cudaStream_t s, double* d_mean) {
    int grid = glm_grid(c.n);
    int nv = 2 + (int)c.q;
    IHTB_LAUNCH(k_score, grid, GLM_THREADS, 0, s, c.n, c.q, c.Z, c.xb, c.zc, c.mu, c.y, c.w, c.dist, c.link, c.nb_r,
                c.r, c.part, c.scal, c.done, d_mean);
    if (!c.done) IHTB_LAUNCH(k_finalize, (unsigned)ceil_div(nv, 4), 128, 0, s, c.part, grid, nv, c.scal, d_mean, c.n);
}
void glm_stepsize(GlmCtx& c, const double* d_d2, const double* d_xs, cudaStream_t s, const double* d_d2mask,
                  double* d_out) {
    int grid = glm_grid(c.n);
    IHTB_LAUNCH(k_stepsize, grid, GLM_THREADS, 0, s, c.n, c.q, c.Z, d_d2, d_d2mask, d_xs, c.xb, c.zc, c.mu, c.w, c.dist,
                c.link, c.nb_r, c.part, d_out ? d_out : c.scal, c.done);
    if (!c.done) IHTB_LAUNCH(k_finalize, 1, 32, 0, s, c.part, grid, 1, d_out ? d_out : c.scal);
}
void glm_sum2(GlmCtx& c, const double* a, const double* b, cudaStream_t s) {
    int grid = glm_grid(c.n);
    IHTB_LAUNCH(k_sum2, grid, GLM_THREADS, 0, s, c.n, a, b, c.part);
    IHTB_LAUNCH(k_finalize, 1, 64, 0, s, c.part, grid, 2, c.scal);
}
void glm_ssq2(GlmCtx& c, const double* a, double ma, const double* b, double mb, cudaStream_t s) {
    int grid = glm_grid(c.n);
    IHTB_LAUNCH(k_ssq2, grid, GLM_THREADS, 0, s, c.n, a, ma, b, mb, c.part);
    IHTB_LAUNCH(k_finalize, 1, 64, 0, s, c.part, grid, 2, c.scal);
}
void glm_set_weights(GlmCtx& c, const uint8_t* d_mask, cudaStream_t s) {
    int grid = glm_grid(c.n);
    IHTB_LAUNCH(k_set_weights, grid, GLM_THREADS, 0, s, c.n, d_mask, c.y, c.w, c.part);
    IHTB_LAUNCH(k_finalize, 1, 64, 0, s, c.part, grid, 2, c.scal);
}

}  // namespace ihtb
