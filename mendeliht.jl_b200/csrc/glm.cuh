// GLM scalar formulas (GLM.jl 1.x / Distributions.jl 0.25; call sites reference src/utilities.jl:32-43,56,80,130,402,749)
#pragma once
#include "common.cuh"
#include <math.h>

namespace ihtb {

constexpr int GLM_MAX_BLOCKS = 1024;

#define IHTB_HDI __host__ __device__ __forceinline__

IHTB_HDI double glm_xlogy(double x, double y) { return (x == 0.0 && !isnan(y)) ? 0.0 : x * log(y); }

IHTB_HDI double glm_linkinv(int link, double eta) {
    switch (link) {
        case IHTB_LINK_IDENTITY: return eta;
        case IHTB_LINK_LOGIT: return 1.0 / (1.0 + exp(-eta));
        case IHTB_LINK_LOG: return exp(eta);
        case IHTB_LINK_PROBIT: return 0.5 * (1.0 + erf(eta / 1.4142135623730951));
        case IHTB_LINK_CLOGLOG: return -expm1(-exp(eta));
        case IHTB_LINK_CAUCHIT: return 0.5 + atan(eta) / 3.141592653589793;
        case IHTB_LINK_SQRT: return eta * eta;
        case IHTB_LINK_INVERSE: return 1.0 / eta;
        case IHTB_LINK_INVSQ: return 1.0 / sqrt(eta);
    }
    return NAN;
}

IHTB_HDI double glm_mueta(int link, double eta) {
    switch (link) {
        case IHTB_LINK_IDENTITY: return 1.0;
        case IHTB_LINK_LOGIT: {
            double e = exp(-fabs(eta));
            double f = 1.0 + e;
            return e / (f * f);
        }
        case IHTB_LINK_LOG: return exp(eta);
        case IHTB_LINK_PROBIT: return exp(-0.5 * eta * eta) / 2.5066282746310002;
        case IHTB_LINK_CLOGLOG: return exp(eta) * exp(-exp(eta));
        case IHTB_LINK_CAUCHIT: return 1.0 / (3.141592653589793 * (1.0 + eta * eta));
        case IHTB_LINK_SQRT: return 2.0 * eta;
        case IHTB_LINK_INVERSE: return -1.0 / (eta * eta);
        case IHTB_LINK_INVSQ: {
            double m = 1.0 / sqrt(eta);
            return -(m * m * m) / 2.0;
        }
    }
    return NAN;
}

IHTB_HDI double glm_var(int dist, double mu, double r) {
    switch (dist) {
        case IHTB_NORMAL: return 1.0;
        case IHTB_BERNOULLI: return mu * (1.0 - mu);
        case IHTB_POISSON: return mu;
        case IHTB_NEGBIN: return mu * (1.0 + mu / r);
    }
    return NAN;
}

IHTB_HDI double glm_devresid(int dist, double y, double mu, double r) {
    switch (dist) {
        case IHTB_NORMAL: {
            double d = y - mu;
            return d * d;
        }
        case IHTB_BERNOULLI:
            if (y == 1.0) return -2.0 * log(mu);
            if (y == 0.0) return -2.0 * log1p(-mu);
            return 2.0 * (glm_xlogy(y, y / mu) + glm_xlogy(1.0 - y, (1.0 - y) / (1.0 - mu)));
        case IHTB_POISSON: return 2.0 * (glm_xlogy(y, y / mu) - (y - mu));
        case IHTB_NEGBIN: {
            double v = 2.0 * (glm_xlogy(y, y / mu) + glm_xlogy(y + r, (mu + r) / (y + r)));
            return mu == 0.0 ? NAN : v;
        }
    }
    return NAN;
}

// log density without the dispersion-dependent part (Normal is closed-form on the host from the deviance)
IHTB_HDI double glm_logpdf_nophi(int dist, double y, double mu, double r) {
    switch (dist) {
        case IHTB_BERNOULLI: return (y == 1.0) ? log(mu) : log(1.0 - mu);
        case IHTB_POISSON: return glm_xlogy(y, mu) - mu - lgamma(y + 1.0);
        case IHTB_NEGBIN: {
            double p = r / (mu + r);
            // logbeta(r, y+1) = lgamma(r) + lgamma(y+1) - lgamma(r+y+1)
            return r * log(p) + y * log1p(-p) - log(y + r) - (lgamma(r) + lgamma(y + 1.0) - lgamma(r + y + 1.0));
        }
    }
    return 0.0;
}

// device pointers of one univariate fit, as the GLM kernels see them
struct GlmCtx {
    int64_t n, q;
    const double* Z;   // n x q column-major
    const double* y;
    double* w;         // cv_wts
    double* xb;
    double* zc;
    double* mu;
    double* r;
    double* part;      // GLM_MAX_BLOCKS * (2 + q) partial sums
    double* scal;      // finalized sums
    int dist, link;
    double nb_r;
    // Tickets of the in-kernel finalisation (one per model of a batched launch, zero between launches): the CTA that draws
    // the last ticket adds the per-CTA partial sums itself -- same order as k_finalize -- instead of a second launch.
    // NULL: separate k_finalize launches (contexts built ad hoc, e.g. mvfit.cu's init_beta).
    unsigned* done = nullptr;
};

void glm_mu(GlmCtx& c, const double* d_c, int add_zc, cudaStream_t s);        // scal: dev, lp, sum w
void glm_mu_batched(GlmCtx& c, const double* d_cM, int M, double* xbM, double* zcM, double* muM, double* d_partM,
                    double* d_scalM, cudaStream_t s);                           // d_scalM[3m..]: dev, lp, sum w of model m
void glm_mean_from_sum(GlmCtx& c, double* d_mean, cudaStream_t s);
// device-side choice among the M candidate models of a step (d_pick[0] = winner, d_pick[1 + m] = loglikelihoods) and
// copy of the winner's xb / zc / mu into the fit's vectors; coefficients / covariate mask of the winner's support
void glm_pick_model(GlmCtx& c, const double* d_scalM, int M, double old_logl, int max_step, double* d_pick,
                    const double* xbM, const double* zcM, const double* muM, cudaStream_t s);
void glm_winner_coef(const double* d_pick, const double* d_coefM, int64_t U, const double* d_df_uni, double* d_coef_out,
                     const double* d_cM, int64_t q, double* d_mask_out, cudaStream_t s);             // d_mean[0] = scal[0] / n
// r, sums [sum r, sum |r|, df2[q]]; d_mean (optional) receives mean(r) = sum r / n
void glm_score(GlmCtx& c, cudaStream_t s, double* d_mean = nullptr);                                      // scal: sum r, sum |r|, df2[q]
// scal[0] (or *d_out) = sum of squares of sqrt(W) (xs + Z (d2 .* d2mask)); d2mask may be NULL
void glm_stepsize(GlmCtx& c, const double* d_d2, const double* d_xs, cudaStream_t s, const double* d_d2mask = nullptr,
                  double* d_out = nullptr);
void glm_sum2(GlmCtx& c, const double* a, const double* b, cudaStream_t s);
void glm_ssq2(GlmCtx& c, const double* a, double ma, const double* b, double mb, cudaStream_t s);
void init_beta_products(GlmCtx& c, double* d_wy, cudaStream_t s);             // d_wy = w .* y
void init_beta_solve(GlmCtx& c, int64_t p, const double* W1, const double* W2, const double* Wm, const double* Y1,
                     const double* Y2, const double* Ym, double N, double SY, const double* mu, const double* sinv,
                     int impute, double* d_beta, cudaStream_t s);                   // scal[0] = sum of intercepts
// dense handles: the same regressions from per-column sums of w x, w x^2 and w y x
void init_beta_solve_moments(GlmCtx& c, int64_t p, const double* SX, const double* SXX, const double* SXY, double N,
                             double SY, double* d_beta, cudaStream_t s);
void init_beta_cov_sums(GlmCtx& c, cudaStream_t s);                               // scal[3(l-1)+{0,1,2}]
void glm_set_weights(GlmCtx& c, const uint8_t* d_mask, cudaStream_t s);        // scal: sum w, sum y*w

}  // namespace ihtb
