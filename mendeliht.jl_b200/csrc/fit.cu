// Univariate IHT driver: the whole fit_iht! loop (reference src/fit.jl:145-263) runs inside one C call.
// O(n), O(p) and O(np) work is on the device; the k-sparse model (b, b0, best_b, supports, c) and the loop control
// live on the host, which reads back a handful of scalars per iteration.
//
// Reference function -> where it is here
//   init_iht_indices!  src/utilities.jl:366-438  -> ihtb_fit::init
//   fit_iht!           src/fit.jl:145-207        -> ihtb_fit::run
//   iht_one_step!      src/fit.jl:213-263        -> ihtb_fit::one_step
//   iht_stepsize!      src/utilities.jl:722-764  -> ihtb_fit::stepsize   (x_support + k_stepsize)
//   _iht_gradstep!     src/utilities.jl:252-280  -> ihtb_fit::gradstep   (topk_candidates + xt_gather + host top-k)
//   update_xb!/update_mu!/loglikelihood          -> ihtb_fit::update_xb / glm_update (k_glm_mu)
//   score!             src/utilities.jl:126-135  -> ihtb_fit::score_and_sweep (k_score + sweep)
//   save_prev!/check_convergence/backtrack!/save_best_model!  -> same names below
//   pve                src/pve.jl:31-33          -> ihtb_fit::compute_pve
#include "glm.cuh"
#include "topk.cuh"
#include "comm.cuh"
#include "debias.cuh"
#include "groups.cuh"
#include "pairer.cuh"
#include <algorithm>
#include <chrono>
#include <cmath>
#include <memory>
#include <mutex>
#include <string.h>
#include <unordered_map>

namespace ihtb {
void sweep_xt_v_with_means(const ihtb_geno* g, const double* dV, const double* vbar_host, int64_t m, double* dOut,
                           int mode, cudaStream_t s, void* scratch_any, float* sweep_ms, double* d_l2 = nullptr,
                           const TopkFuse* tf = nullptr);
void* sweep_scratch_create();
void sweep_scratch_destroy(void* p);
void sweep_class_sums(const ihtb_geno* g, const double* d_v, double* d_w1, double* d_w2, double* d_wm, cudaStream_t s,
                      void* scratch_any);
}  // namespace ihtb

using namespace ihtb;

// worst-case absolute error of the FAST sweep's sum_i dosage_ij u_i, as a multiple of ||u||_1 :
// 1 rounding of u to FP32 + 3 adds in the table (4 with the ternary tiles: five dosages per byte) + 3 adds per word +
// 5 levels of the pairwise tree over a chunk's 32 words (butterfly or per-lane, sweep_lut.cu) = 13 roundings of at most
// 2^-24 relative on partial sums bounded by 2*||u||_1 (dosage <= 2)
// ->  13 * 2^-24 * 2 = 1.55e-6 ; we use 2^-18 = 3.8e-6 (2.5x margin).  The FP64 cross-slab sums add < 1e-13.
static const double kFastBound = 1.0 / 262144.0;
static const double kExactBound = 1e-13;
// PAIR sweep (half2 tables, sweep_lut.cu): one FP16 rounding per table entry + two levels of HADD2 per packed word, each
// at most 2^-11 of a partial sum bounded by A_j = sum_i g_ij |u_i| <= sqrt(sum_i g_ij^2) ||u||_2 (Cauchy-Schwarz); FP32
// conversions and sums, the FP32 rounding of u and FP16 subnormals add less than 2^-16 of that.  The bound is
// kPairBound * ||u||_2 * sgn_j with the per-column scale sgn_j = sinv_j * max(sqrt(sum_i g_ij^2), 1) of the handle.
static const double kPairBound = 3.1 / 2048.0;

struct ihtb_fit {
    const ihtb_geno* g = nullptr;
    int device = 0;
    int64_t n = 0, p = 0, q = 0;          // p = local SNP columns
    // SNP-sharded fits: this rank owns global columns [j0, j0 + p); the k-sparse model, y, z and every n-vector are
    // replicated; partial X*beta is all-reduced and top-k candidates are all-gathered (SURVEY.md 8e)
    ihtb_comm* comm = nullptr;
    int64_t j0 = 0, p_global = 0;
    std::vector<int64_t> shard_j0;        // j0 of every rank
    DBuf<int64_t> d_selall, d_pack, d_packall;
    HBuf<int64_t> h_selall, h_packall;
    int capx = 512;                       // per-rank capacity of the (index, value) candidate exchange
    ihtb_cfg cfg{};
    cudaStream_t s = nullptr;
    std::vector<uint8_t> zkeep;
    int zkeepn = 0;
    int cap = 4096;

    // device state
    DBuf<unsigned> d_done;
    DBuf<double> d_y, d_z, d_w, d_xb, d_zc, d_mu, d_r, d_xs, d_dfa, d_part, d_scal, d_small, d_coef, d_gout,
        d_vbar;
    DBuf<uint8_t> d_mask;
    DBuf<uint32_t> d_keyL, d_keyU;
    DBuf<int> d_hist;
    DBuf<int64_t> d_sel;   // [TopkState (2 x int64) | cand[cap]]
    DBuf<int64_t> d_idx, d_cols;
    HBuf<double> h_scal, h_gout;
    HBuf<int64_t> h_sel;
    void* sweep_scratch = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, tm0 = nullptr, tm1 = nullptr;
    bool sweep_pending = false;
    // one_step_fused: the score phase is enqueued before the host knows which candidate model won
    struct FusedStep {
        std::vector<int64_t> uni_loc;     // this rank's columns of the union of the candidate supports (local indices)
        size_t maxsupp = 0;               // largest candidate support
        int M = 0;
        int winner = -1;
    };
    FusedStep* fz = nullptr;
    DBuf<double> d_pick;
    HBuf<double> h_pick;
    // cross-validation farm: two fits of one device share their sweeps (pairer.cuh); null = every sweep alone
    SweepPairer* pairer = nullptr;
    int pair_slot = 0;
    double sweep_coef = kFastBound;       // error-bound coefficient of the LAST sweep (what the selection must assume)
    GlmCtx glm{};
    TopkCtx tk{};

    // host model state (k-sparse)
    std::vector<int64_t> idx, idx0, best_idx;
    std::vector<double> b, b0, best_b;
    std::vector<double> c, c0, best_c, df2, h_y, h_mu;
    std::vector<uint8_t> idc, idc0;
    std::unordered_map<int64_t, double> df_exact;
    // prior weights (src/data_structures.jl:36): host copy over all p_global SNPs, device copy of this rank's columns
    std::vector<double> wt;
    DBuf<double> d_wt;
    double w_at(int64_t j) const { return wt.empty() ? 1.0 : wt[(size_t)j]; }
    void set_weights(const double* w) {
        if (!w) { wt.clear(); tk.wt = nullptr; return; }
        for (int64_t j = 0; j < p_global; ++j)
            IHTB_CHECK(w[j] > 0.0 && std::isfinite(w[j]), IHTB_EDOMAIN, "weights must be positive and finite");
        wt.assign(w, w + p_global);
        if (d_wt.n < (size_t)p) d_wt.alloc((size_t)p);
        IHTB_CUDA(cudaMemcpyAsync(d_wt.p, wt.data() + j0, (size_t)p * sizeof(double), cudaMemcpyHostToDevice, s));
        sync();
        tk.wt = d_wt.p;
    }
    std::vector<int64_t> cand_cache;      // candidate columns of the last sweep (global indices, sorted)
    bool df_sparse = false;
    std::vector<int64_t> dfs_idx;
    std::vector<double> dfs_val;
    double rbar = 0.0, bound = 0.0, sum_w = 0.0, sum_wy = 0.0, last_dev = 0.0, denom_next = 0.0;
    bool denom_ready = false;
    bool inited = false;

    // statistics
    int64_t n_sweeps = 0, n_backtracks = 0, n_cand_iter = 0, n_pair_overflow = 0;
    int last_count = 0;                    // candidates the last selection found (sizes the next re-scoring launch)
    double sweep_ms_total = 0.0;
    double pve = 0.0;

    ~ihtb_fit() {
        if (sweep_scratch) sweep_scratch_destroy(sweep_scratch);
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        if (tm0) cudaEventDestroy(tm0);
        if (tm1) cudaEventDestroy(tm1);
        if (s) cudaStreamDestroy(s);
    }

    // ------------------------------------------------------------------------------------------
    void sync() { IHTB_CUDA(cudaStreamSynchronize(s)); }
    void readback_scal(int nv) {
        IHTB_CUDA(cudaMemcpyAsync(h_scal.p, d_scal.p, nv * sizeof(double), cudaMemcpyDeviceToHost, s));
        sync();
    }
    template <typename T>
    void upload(T* dst, const T* src, size_t count) {
        if (count) IHTB_CUDA(cudaMemcpyAsync(dst, src, count * sizeof(T), cudaMemcpyHostToDevice, s));
    }

    bool is_local(int64_t j) const { return j >= j0 && j < j0 + p; }
    int nranks() const { return comm ? comm->nranks : 1; }

    // d_out = x[:, cols] * coef over the GLOBAL column list: local partial + all-reduce over the shards
    void support_matvec(const std::vector<int64_t>& cols, const std::vector<double>& coef, double* d_out) {
        std::vector<int64_t> ii; std::vector<double> vv;
        for (size_t t = 0; t < cols.size(); ++t)
            if (coef[t] != 0.0 && is_local(cols[t])) { ii.push_back(cols[t] - j0); vv.push_back(coef[t]); }
        if (!ii.empty()) {
            upload(d_idx.p, ii.data(), ii.size());
            upload(d_coef.p, vv.data(), vv.size());
        }
        support_matvec_dev(ii.empty() ? nullptr : d_idx.p, (int64_t)ii.size(), d_coef.p, d_out);
    }

    // same with the local index / coefficient lists already on the device.  Sharded fits with the peer-memory path:
    // the partial vector is produced straight into every rank's slot and reduced locally (p2p.cu); otherwise NCCL.
    void support_matvec_dev(const int64_t* d_idx_loc, int64_t k_loc, const double* d_coef_loc, double* d_out) {
        support_matvec_dev_m(d_idx_loc, k_loc, d_coef_loc, 1, d_out);
    }
    // m models at once (coef is k_loc x m column-major, d_out is n x m): short vectors take the fused push-all path
    // (m == 1), long ones are produced straight into this rank's partial area and reduced in two phases (p2p.cu)
    void support_matvec_dev_m(const int64_t* d_idx_loc, int64_t k_loc, const double* d_coef_loc, int m, double* d_out) {
        const size_t cnt = (size_t)n * (size_t)m;
        if (!comm) {
            if (k_loc > 0) x_support(g, d_idx_loc, k_loc, d_coef_loc, m, d_out, s);
            else IHTB_CUDA(cudaMemsetAsync(d_out, 0, cnt * sizeof(double), s));
            return;
        }
        if (m == 1 && p2p_pushall_ok(comm, cnt)) {
            if (k_loc > 0) x_support_push(g, d_idx_loc, k_loc, d_coef_loc, comm, s);
            else p2p_push(comm, nullptr, cnt, s);
            p2p_reduce(comm, d_out, cnt, s);
            return;
        }
        if (p2p_mapped(comm) && cnt <= comm->red_cap) {
            double* part = p2p_partial_ptr(comm);
            if (k_loc > 0) x_support(g, d_idx_loc, k_loc, d_coef_loc, m, part, s);
            else IHTB_CUDA(cudaMemsetAsync(part, 0, cnt * sizeof(double), s));
            p2p_allreduce_2phase(comm, cnt, d_out, s);
            return;
        }
        if (k_loc > 0) x_support(g, d_idx_loc, k_loc, d_coef_loc, m, d_out, s);
        else IHTB_CUDA(cudaMemsetAsync(d_out, 0, cnt * sizeof(double), s));
        comm_allreduce_sum_f64(comm, d_out, cnt, s);
    }

    // ---- update_xb! genetic part: xb = x[:, idx] * b[idx]  (src/utilities.jl:95-111) ------------
    void update_xb() { support_matvec(idx, b, d_xb.p); }

    // ---- zc = Z c, clamp, mu = linkinv, deviance, loglikelihood (src/utilities.jl:9-20,52-61,74-82,113-117) ----
    double glm_update(int add_zc) {
        upload(d_small.p, c.data(), (size_t)q);
        glm_mu(glm, d_small.p, add_zc, s);
        readback_scal(3);
        double dev = h_scal.p[0], lp = h_scal.p[1], sw = h_scal.p[2];
        last_dev = dev;
        if (cfg.dist == IHTB_NORMAL) {
            double phi = dev / (double)n;               // deviance / length(y), even under CV masks
            double sigma = std::sqrt(phi);
            return -0.5 * (dev / phi) - sw * (0.5 * std::log(2.0 * M_PI) + std::log(sigma));
        }
        return lp;
    }

    // ---- mle_for_r: nuisance parameter of the negative binomial (src/utilities.jl:141-247) ---------------
    // n-vector loops on the host (mu and y are copied back); the loglikelihood of the Newton line search runs on
    // the device through glm_update.  Like the reference, the estimate persists in the fit variable (v.d).
    static double digamma(double x) {
        double r = 0.0;
        while (x < 6.0) { r -= 1.0 / x; x += 1.0; }
        double f = 1.0 / (x * x);
        return r + std::log(x) - 0.5 / x -
               f * (1.0 / 12 - f * (1.0 / 120 - f * (1.0 / 252 - f * (1.0 / 240 - f * (1.0 / 132)))));
    }
    static double trigamma(double x) {
        double r = 0.0;
        while (x < 6.0) { r += 1.0 / (x * x); x += 1.0; }
        double f = 1.0 / (x * x);
        return r + 1.0 / x + f / 2 + f / x * (1.0 / 6 - f * (1.0 / 30 - f * (1.0 / 42 - f * (1.0 / 30))));
    }
    void fetch_mu() {
        h_mu.resize((size_t)n);
        IHTB_CUDA(cudaMemcpyAsync(h_mu.data(), d_mu.p, n * sizeof(double), cudaMemcpyDeviceToHost, s));
        sync();
    }
    double nb_logl(double r) {            // negbin_loglikelihood(r): v.d = NegativeBinomial(r); loglikelihood(v)
        glm.nb_r = r;
        return glm_update(1);
    }
    void mle_for_r() {
        fetch_mu();
        const std::vector<double>& y = h_y;
        double r = glm.nb_r;
        if (cfg.est_r == 1) {             // update_r_MM (:158-173)
            double num = 0.0, den = 0.0;
            for (int64_t i = 0; i < n; ++i) {
                for (int64_t j = 0; j <= (int64_t)y[i] - 1; ++j) num += r / (r + (double)j);
                den += std::log(r / (r + h_mu[i]));
            }
            glm.nb_r = -num / den;
            return;
        }
        // update_r_newton (:180-247)
        auto d1 = [&](double rr) {
            double a = 0.0;
            for (int64_t i = 0; i < n; ++i)
                a += -(y[i] + rr) / (h_mu[i] + rr) - std::log(h_mu[i] + rr) + 1.0 + std::log(rr) + digamma(rr + y[i]) -
                     digamma(rr);
            return a;
        };
        auto d2 = [&](double rr) {
            double a = 0.0;
            for (int64_t i = 0; i < n; ++i)
                a += (y[i] + rr) / ((h_mu[i] + rr) * (h_mu[i] + rr)) - 2.0 / (h_mu[i] + rr) + 1.0 / rr +
                     trigamma(rr + y[i]) - trigamma(rr);
            return a;
        };
        double new_r = 1.0, stepsize = 1.0;
        for (int it = 0; it < 100; ++it) {
            double dx = d1(r), dx2 = d2(r);
            double increment = dx2 < 0 ? dx / dx2 : dx;
            new_r = r - stepsize * increment;
            double old_logl = nb_logl(r);
            for (int j = 0; j < 20; ++j) {
                if (new_r <= 0) {
                    stepsize /= 2; new_r = r - stepsize * increment;
                } else {
                    double new_logl = nb_logl(new_r);
                    if (old_logl >= new_logl) { stepsize /= 2; new_r = r - stepsize * increment; }
                    else break;
                }
            }
            if (std::fabs(r - new_r) <= 1e-6) { glm.nb_r = new_r; return; }
            r = new_r;
        }
        glm.nb_r = r;
    }
    // update_mu!; [mle_for_r]; loglikelihood  (src/fit.jl:226-240, src/utilities.jl:966-972)
    double mu_r_logl() {
        double l = glm_update(1);
        if (cfg.est_r != 0) {
            mle_for_r();
            l = glm_update(1);
        }
        return l;
    }

    // ---- exact df_j for a list of columns (cached until the next sweep) --------------------------
    // exchange = false (sharded fits): only this rank's columns are computed; the others arrive later piggy-backed on
    // a collective that is needed anyway (stepsize all-reduce / candidate all-gather)
    void exact_df(const std::vector<int64_t>& cols, bool exchange = true) {
        std::vector<int64_t> need;
        for (int64_t j : cols)
            if (!df_exact.count(j) && (exchange || is_local(j))) need.push_back(j);
        if (need.empty()) { if (!exchange) sync(); return; }
        IHTB_CHECK((int64_t)need.size() <= (int64_t)d_cols.n, IHTB_ENUMERIC, "too many columns to re-score");
        // columns of other shards are marked -1: the kernel writes 0 for them and the all-reduce fills them in
        std::vector<int64_t> loc(need.size());
        for (size_t t = 0; t < need.size(); ++t) loc[t] = is_local(need[t]) ? need[t] - j0 : -1;
        upload(d_cols.p, loc.data(), loc.size());
        xt_gather2(g, d_cols.p, (int64_t)need.size(), nullptr, 0, d_r.p, 1, d_vbar.p, d_gout.p, s,
                   false);                              // d_vbar = mean(r), set by score
        if (exchange) comm_allreduce_sum_f64(comm, d_gout.p, need.size(), s);
        IHTB_CUDA(cudaMemcpyAsync(h_gout.p, d_gout.p, need.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
        sync();
        for (size_t t = 0; t < need.size(); ++t) df_exact[need[t]] = h_gout.p[t];
        n_cand_iter += (int64_t)need.size();
    }

    // ---- score! : r, df2 = Z'r, df = X'r (src/utilities.jl:126-135) ------------------------------
    // One host round trip for everything that follows a sweep.  Enqueued back to back on the stream:
    //   k_score -> mean(r) -> sweep -> eta-independent candidate selection (top-(k+|supp|) of |df| with the sweep's
    //   error bound, computed on the device) -> exact FP64 re-scoring of those candidates and of the current support
    //   [-> sharded: one all-gather of (index, exact value) pairs].
    // The top-k of |b0 + eta*df| always lies in supp(b0) plus the k largest |df_j| outside it, for ANY eta, so the
    // gradient step and all its backtracks are then pure host work on ~2k exact values.
    void score_and_sweep() {
        glm_score(glm, s, d_vbar.p);                         // scal: sum r, sum |r|, df2[q]; d_vbar[0] = scal[0] / n
        IHTB_CUDA(cudaMemcpyAsync(h_scal.p, d_scal.p, (2 + q) * sizeof(double), cudaMemcpyDeviceToHost, s));
        IHTB_CUDA(cudaEventRecord(ev0, s));
        sweep_coef = geno_bound_coef(g, cfg.sweep_mode == IHTB_SWEEP_FAST ? kFastBound : kExactBound);
        const double t_sw = now();
        if (pairer && cfg.sweep_mode == IHTB_SWEEP_FAST) {
            IHTB_CHECK(!grouped() && !comm, IHTB_EUNSUPPORTED, "paired sweeps serve plain single-device fits only");
            if (pairer->sweep(pair_slot, g, d_r.p, d_vbar.p, d_dfa.p, s, sweep_scratch)) {
                sweep_coef = kPairBound;
                // ||r - mean||_2 of this fit travels back with the other score sums
                IHTB_CUDA(cudaMemcpyAsync(h_scal.p + 3 + q, pairer->d_l2 + pair_slot, sizeof(double), cudaMemcpyDeviceToHost, s));
            }
        } else if (cfg.k > 0 && !(grouped() && !init_plain)) {
            // the epilogue also runs the first stage of the candidate selection (keys of |df| with this sweep's error bound,
            // first digit histogram); select_rescore continues with topk_candidates_absdf_finish
            const TopkFuse tf = topk_absdf_fuse_begin(tk, geno_bound_scale(g), d_scal.p, sweep_coef);
            sweep_xt_v_with_means(g, d_r.p, d_vbar.p, 1, d_dfa.p, cfg.sweep_mode, s, sweep_scratch, nullptr, nullptr, &tf);
        } else {
            sweep_xt_v_with_means(g, d_r.p, d_vbar.p, 1, d_dfa.p, cfg.sweep_mode, s, sweep_scratch, nullptr);
        }
        IHTB_CUDA(cudaEventRecord(ev1, s));
        ++n_sweeps;
        const double t_sel = now();
        dbg[0] += t_sel - t_sw;
        select_rescore(/*rerun=*/false);
        dbg[1] += now() - t_sel;
    }

    // Candidate selection + exact re-scoring for the CURRENT idx against the last sweep's df (see score_and_sweep).
    // rerun = true: called a second time for the same sweep (init_beta changes the support after the sweep); the
    // score sums are no longer on the device, so the host copy of the error bound is used and no scalars are read.
    void select_rescore(bool rerun) {
        if (grouped() && !init_plain) {
            select_groups(rerun);
            if (!rerun) finish_sweep_scalars(sweep_coef);
            return;
        }
        df_exact.clear(); cand_cache.clear();
        df_sparse = false;
        const double coef = sweep_coef;
        // (column, exact df) of every candidate; only the ones that survive the trim below enter df_exact -- a paired
        // sweep may list thousands, and a hash-map insertion per candidate would cost more than the sweep saves
        std::vector<std::pair<int64_t, double>> cvals;
        // this rank's part of the current support (local indices); fused step: of the union of the candidate models'
        // supports (already on the device in d_idx), since the winner is only known after the read-back
        const bool fused = fz != nullptr && !rerun;
        std::vector<int64_t> supp_loc;
        if (fused) supp_loc = fz->uni_loc;
        else
            for (int64_t j : idx)
                if (is_local(j)) supp_loc.push_back(j - j0);
        const int nsupp = (int)supp_loc.size();
        const int64_t* d_supp = fused ? d_idx.p : d_cols.p;
        int glaunch = 0;
        if (cfg.k > 0) {
            const int64_t ksel = cfg.k + (int64_t)(fused ? fz->maxsupp : idx.size());
            const bool paired = coef == kPairBound;        // L2 bound over the handle's sgn scale (see kPairBound)
            if (tk.fused_hist) topk_candidates_absdf_finish(tk, ksel, s);      // first stage done by the sweep epilogue
            else
                topk_candidates_absdf(tk, d_dfa.p, paired ? g->sgn.p : geno_bound_scale(g), rerun ? nullptr : d_scal.p, coef, ksel, s,
                                      bound, (paired && !rerun) ? pairer->d_l2 + pair_slot : nullptr);
            // slots re-scored without a second round trip; the looser bound of a PAIR sweep admits more near-threshold columns
            // (sized from the previous iteration's count there)
            const int64_t want = sweep_coef == kPairBound ? std::max<int64_t>(ksel + 1024, last_count + last_count / 4 + 256)
                                                          : ksel + 64;
            glaunch = (int)std::min<int64_t>(comm ? capx / 2 : cap, want);
        }
        if (nsupp && !fused) upload(d_cols.p, supp_loc.data(), supp_loc.size());
        // candidates (slots beyond the count hold -1) and the current support re-scored exactly in ONE launch
        xt_gather2(g, tk.cand, glaunch, d_supp, nsupp, d_r.p, 1, d_vbar.p, d_gout.p, s);
        // the next iteration's step-size denominator ||sqrt(W) (X[:,idx] df[idx] + Z[:,idc] df2[idc])||^2 needs nothing
        // from the host either: the support's exact df values are in d_gout, df2 is in d_scal (src/utilities.jl:728-756)
        denom_ready = false;
        if (!rerun) {
            if (fused) {
                // the winner's support is a subset of the union: zero the other coefficients on the device
                glm_winner_coef(d_pick.p, d_coefM.p, nsupp, d_gout.p + glaunch, d_coef.p, d_cM.p, q, d_small.p + q, s);
                support_matvec_dev(d_supp, nsupp, d_coef.p, d_xs.p);
                IHTB_CUDA(cudaMemcpyAsync(h_pick.p, d_pick.p, (size_t)(1 + fz->M) * sizeof(double), cudaMemcpyDeviceToHost, s));
                IHTB_CUDA(cudaMemcpyAsync(h_scalM.p, d_scalM.p, (size_t)(3 * fz->M) * sizeof(double), cudaMemcpyDeviceToHost, s));
            } else {
                support_matvec_dev(d_supp, nsupp, d_gout.p + glaunch, d_xs.p);
                std::vector<double> mask((size_t)q);
                for (int64_t l = 0; l < q; ++l) mask[l] = idc[l] ? 1.0 : 0.0;
                upload(d_small.p + q, mask.data(), (size_t)q);
            }
            glm_stepsize(glm, d_scal.p + 2, d_xs.p, s, d_small.p + q, d_scal.p + 2 + q);
            IHTB_CUDA(cudaMemcpyAsync(h_scal.p + 2 + q, d_scal.p + 2 + q, sizeof(double), cudaMemcpyDeviceToHost, s));
            denom_ready = true;
        }
        if (!comm) {
            IHTB_CUDA(cudaMemcpyAsync(h_sel.p, d_sel.p, (2 + glaunch) * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
            IHTB_CUDA(cudaMemcpyAsync(h_gout.p, d_gout.p, (glaunch + nsupp) * sizeof(double), cudaMemcpyDeviceToHost, s));
            sync();
            const double t_host = now();
            struct Acc { double& a; double t0; ~Acc() { a += now() - t0; } } acc_host{dbg[2], t_host};
            if (fused) adopt_winner();
            const TopkState* st = reinterpret_cast<const TopkState*>(h_sel.p);
            const int count = cfg.k > 0 ? st->count : 0;
            dbg[3] += (double)std::min(count, glaunch);
            if (count > cap && coef == kPairBound && !rerun) {
                // the looser bound of the PAIR sweep admits more columns than can be re-scored: sweep this residual
                // alone with the FP32 tables and select again (results never depend on which sweep served them)
                ++n_pair_overflow;
                sweep_coef = kFastBound;
                sweep_xt_v_with_means(g, d_r.p, d_vbar.p, 1, d_dfa.p, IHTB_SWEEP_FAST, s, sweep_scratch, nullptr);
                IHTB_CUDA(cudaEventRecord(ev1, s));
                select_rescore(false);
                return;
            }
            IHTB_CHECK(count <= cap, IHTB_ENUMERIC,
                       "degenerate projection: more than " + std::to_string(cap) +
                           " entries lie within the sweep error bound of the k-th largest |gradient|");
            last_count = count;
            cvals.reserve((size_t)count);
            for (int t = 0; t < std::min(count, glaunch); ++t) cvals.push_back({h_sel.p[2 + t], h_gout.p[t]});
            for (int t = 0; t < nsupp; ++t) df_exact[supp_loc[t] + j0] = h_gout.p[glaunch + t];
            if (count > glaunch) {                       // rare: many near-ties; fetch and re-score the remainder
                IHTB_CUDA(cudaMemcpyAsync(h_sel.p, d_sel.p, (2 + count) * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
                sync();
                std::vector<int64_t> rest(h_sel.p + 2 + glaunch, h_sel.p + 2 + count);
                exact_df(rest);
                for (int64_t j : rest) cvals.push_back({j, df_exact.at(j)});
            }
        } else {
            const int nr = nranks();
            const size_t blk = 2 + 2 * (size_t)capx;
            IHTB_CHECK(nsupp <= capx / 2, IHTB_ENUMERIC, "support too large for the sharded candidate exchange");
            pack_sweep_candidates(d_pack.p, reinterpret_cast<const TopkState*>(d_sel.p), tk.cand, glaunch, d_gout.p,
                                  d_supp, nsupp, d_gout.p + glaunch, j0, capx, s);
            comm_allgather_i64(comm, d_pack.p, d_packall.p, blk, s);
            IHTB_CUDA(cudaMemcpyAsync(h_packall.p, d_packall.p, nr * blk * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
            sync();
            if (fused) adopt_winner();
            for (int r = 0; r < nr; ++r) {
                const int64_t* b_ = h_packall.p + (size_t)r * blk;
                IHTB_CHECK(b_[0] <= glaunch, IHTB_ENUMERIC,
                           "degenerate projection: too many local candidates within the sweep error bound");
                const int half = capx / 2;
                auto take = [&](int t, bool is_cand) {
                    const int64_t j = b_[2 + t];
                    if (j < 0) return;
                    double v;
                    memcpy(&v, &b_[2 + capx + t], sizeof(double));
                    if (is_cand) cvals.push_back({j, v});
                    else df_exact[j] = v;
                };
                for (int t = 0; t < (int)b_[0]; ++t) take(t, true);                 // rank r's candidates
                for (int t = 0; t < (int)b_[1]; ++t) take(half + t, false);         // rank r's part of the support
            }
        }
        std::sort(cvals.begin(), cvals.end());
        cvals.erase(std::unique(cvals.begin(), cvals.end(), [](const std::pair<int64_t, double>& x, const std::pair<int64_t, double>& y) {
                        return x.first == y.first; }), cvals.end());
        n_cand_iter += (int64_t)cvals.size();
        // Only the k largest exact |df| OUTSIDE the support can enter P_k(b0 + eta*df) for any eta (the support itself
        // is always a candidate); with R ranks the merged list holds R x (k + |supp|) entries, so trim it once here
        // instead of sorting it in every gradstep/backtrack.  Entries within a relative 1e-12 of the k-th value stay:
        // eta*df may round two nearly equal magnitudes to a tie, which is then broken by index.
        std::vector<char> keep(cvals.size(), 1);
        if ((int64_t)cvals.size() > cfg.k) {
            std::vector<std::pair<double, size_t>> outside;
            outside.reserve(cvals.size());
            for (size_t t = 0; t < cvals.size(); ++t)
                if (!std::binary_search(idx.begin(), idx.end(), cvals[t].first))
                    outside.push_back({std::fabs(cvals[t].second) * w_at(cvals[t].first), t});
            if ((int64_t)outside.size() > cfg.k) {
                std::nth_element(outside.begin(), outside.begin() + (cfg.k - 1), outside.end(),
                                 [](const std::pair<double, size_t>& x, const std::pair<double, size_t>& y) {
                                     return x.first > y.first;
                                 });
                const double thr = outside[(size_t)cfg.k - 1].first * (1.0 - 1e-12);
                std::fill(keep.begin(), keep.end(), 0);
                for (const auto& e : outside)
                    if (e.first >= thr) keep[e.second] = 1;
            }
        }
        for (size_t t = 0; t < cvals.size(); ++t)
            if (keep[t]) {
                cand_cache.push_back(cvals[t].first);             // cvals is sorted by column: so is cand_cache
                df_exact[cvals[t].first] = cvals[t].second;
            }
        if (rerun) return;
        finish_sweep_scalars(coef);
    }

    // host copies of the score sums that travelled back with the candidates
    void finish_sweep_scalars(double coef) {
        float ms = 0.f;
        IHTB_CUDA(cudaEventElapsedTime(&ms, ev0, ev1));
        sweep_ms_total += ms;
        double rsum = h_scal.p[0], rl1 = h_scal.p[1];
        for (int64_t l = 0; l < q; ++l) df2[l] = h_scal.p[2 + l];
        denom_next = h_scal.p[2 + q];
        rbar = rsum / (double)n;
        bound = coef == kPairBound ? coef * h_scal.p[3 + q]  // same value the selection kernel used
                                   : coef * (rl1 + std::fabs(rsum));
    }

    double df_at(int64_t j) const {
        if (df_sparse) {
            auto it = std::lower_bound(dfs_idx.begin(), dfs_idx.end(), j);
            return (it != dfs_idx.end() && *it == j) ? dfs_val[it - dfs_idx.begin()] : 0.0;
        }
        return df_exact.at(j);
    }

    // ---- iht_stepsize! (src/utilities.jl:722-764) -------------------------------------------------
    double stepsize() {
        std::vector<double> coef(idx.size());
        double numer = 0.0;
        for (size_t t = 0; t < idx.size(); ++t) { coef[t] = df_at(idx[t]); numer += coef[t] * coef[t]; }
        if (denom_ready && !df_sparse) {       // denominator already computed behind the sweep (score_and_sweep)
            denom_ready = false;
            for (int64_t l = 0; l < q; ++l)
                if (idc[l]) numer += df2[l] * df2[l];
            double eta = numer / denom_next;
            if (std::isinf(eta) || std::isnan(eta)) eta = 1e-8;
            return eta;
        }
        denom_ready = false;
        support_matvec(idx, coef, d_xs.p);
        std::vector<double> d2((size_t)q);
        for (int64_t l = 0; l < q; ++l) {
            d2[l] = idc[l] ? df2[l] : 0.0;
            if (idc[l]) numer += df2[l] * df2[l];
        }
        upload(d_small.p + q, d2.data(), (size_t)q);
        glm_stepsize(glm, d_small.p + q, d_xs.p, s);
        readback_scal(1);
        double denom = h_scal.p[0];
        double eta = numer / denom;
        if (std::isinf(eta) || std::isnan(eta)) eta = 1e-8;
        return eta;
    }

    static double b_lookup(const std::vector<int64_t>& ii, const std::vector<double>& vv, int64_t j) {
        auto it = std::lower_bound(ii.begin(), ii.end(), j);
        return (it != ii.end() && *it == j) ? vv[it - ii.begin()] : 0.0;
    }

    // ---- _iht_gradstep! : b = P_k(b0 + eta*df), c = c0 + eta*df2 (src/utilities.jl:252-280) --------
    // Ties at the k-th magnitude: lowest position in [b; c] wins (the reference prunes at random, :444-458).
    void gradstep(double eta) {
        if (grouped()) { gradstep_group(eta); return; }
        std::vector<int64_t> cand;
        cand = df_sparse ? dfs_idx : cand_cache;     // chosen once per sweep, exact values already in df_exact
        cand.insert(cand.end(), idx0.begin(), idx0.end());
        std::sort(cand.begin(), cand.end());
        cand.erase(std::unique(cand.begin(), cand.end()), cand.end());

        struct Item { double a; int64_t pos; double v; };
        std::vector<Item> items;
        items.reserve(cand.size() + (size_t)q);
        for (int64_t j : cand) {
            double v = b_lookup(idx0, b0, j) + eta * df_at(j);
            if (!wt.empty()) {          // vectorize!: a = b*w ... unvectorize!: b = a/w (src/utilities.jl:302-304,340-342)
                const double w = wt[(size_t)j], a = v * w;
                items.push_back({std::fabs(a), j, a / w});
            } else {
                items.push_back({std::fabs(v), j, v});
            }
        }
        for (int64_t l = 0; l < q; ++l) {
            c[l] = c0[l] + eta * df2[l];
            if (!zkeep[l]) items.push_back({std::fabs(c[l]), p_global + l, c[l]});
        }
        int64_t k = cfg.k;
        std::sort(items.begin(), items.end(), [](const Item& x, const Item& y) {
            return x.a > y.a || (x.a == y.a && x.pos < y.pos);
        });
        idx.clear(); b.clear();
        // project_k! (:553-559) zeroes the entries BELOW the k-th largest magnitude, so ties at it all survive ...
        const double thr = project_threshold(items, k);
        std::vector<std::pair<int64_t, double>> keep;
        for (size_t t = 0; t < items.size(); ++t) {
            const bool kept = items[t].a >= thr;
            if (items[t].pos >= p_global) {
                if (!kept) c[items[t].pos - p_global] = 0.0;
            } else if (kept && items[t].v != 0.0) {
                keep.push_back({items[t].pos, items[t].v});
            }
        }
        for (int64_t l = 0; l < q; ++l) idc[l] = c[l] != 0.0;
        // ... and _choose! (:444-458) prunes only what exceeds k + zkeepn entries
        choose_prune(keep);
        std::sort(keep.begin(), keep.end());
        for (auto& kv : keep) { idx.push_back(kv.first); b.push_back(kv.second); }
    }

    // threshold of project_k!(x, k + zkeepn) over the candidate entries (kept covariates are +Inf in the reference's
    // vector and never compete): the k-th largest magnitude, 0 when there are fewer than k entries, +Inf for k = 0
    template <typename ItemT>
    static double project_threshold(const std::vector<ItemT>& sorted_items, int64_t k) {
        if (k <= 0) return INFINITY;
        return (int64_t)sorted_items.size() >= k ? sorted_items[(size_t)k - 1].a : 0.0;
    }
    // _choose! (src/utilities.jl:444-458): when ties at the threshold leave more than k + zkeepn non-zero entries
    // (SNPs + covariates, kept covariates counted once: nonzero = |idx| + |idc| - zkeepn), the reference zeroes
    // randomly chosen SNP entries; here (and in the oracle) the smallest magnitudes go first, highest index first
    void choose_prune(std::vector<std::pair<int64_t, double>>& keep) const {
        int64_t nonzero = (int64_t)keep.size() - zkeepn;
        for (int64_t l = 0; l < q; ++l) nonzero += idc[l] ? 1 : 0;
        const int64_t limit = cfg.k + zkeepn;
        if (nonzero <= limit) return;
        std::vector<std::pair<int64_t, double>> byabs = keep;
        std::sort(byabs.begin(), byabs.end(), [](const std::pair<int64_t, double>& x, const std::pair<int64_t, double>& y) {
            return std::fabs(x.second) < std::fabs(y.second) || (std::fabs(x.second) == std::fabs(y.second) && x.first > y.first);
        });
        const size_t excess = std::min<size_t>((size_t)(nonzero - limit), byabs.size());
        for (size_t t = 0; t < excess; ++t) keep.erase(std::find(keep.begin(), keep.end(), byabs[t]));
    }

    // ---- doubly sparse projection (keywords J / k / group; project_group_sparse!, src/utilities.jl:613-679) --------
    std::unique_ptr<GroupCtx> grpctx;          // null: plain top-k projection
    bool init_plain = false;                    // init_iht_indices! with a scalar k projects WITHOUT groups (:417-425)
    bool grouped() const { return (bool)grpctx; }
    void set_groups(const int32_t* group1, int J, const int64_t* ks, int64_t n_groups) {
        if (!group1) { grpctx.reset(); return; }
        IHTB_CHECK(J >= 0, IHTB_EINVAL, "Value of J (max number of groups) must be nonnegative!");
        std::unique_ptr<GroupCtx> gc(new GroupCtx());
        std::vector<double> h_sinv((size_t)p);
        IHTB_CUDA(cudaMemcpy(h_sinv.data(), geno_bound_scale(g), (size_t)p * sizeof(double), cudaMemcpyDeviceToHost));
        gc->build(p, j0, p_global, group1, J, ks, n_groups, cfg.k, h_sinv.data());
        grpctx = std::move(gc);
    }

    // once per sweep: per-group candidate lists (with the sweep's error bound), the groups that can matter, and the
    // exact FP64 df of their candidates and of the current support (groups.cu)
    void select_groups(bool rerun) {
        GroupCtx& gc = *grpctx;
        df_exact.clear(); cand_cache.clear();
        df_sparse = false; denom_ready = false;
        const double coef = sweep_coef;
        group_topk(gc, d_dfa.p, geno_bound_scale(g), rerun ? nullptr : d_scal.p, coef, bound, cfg.k, s);
        const size_t G = (size_t)gc.G, nT = 2 * G + 1;
        const int nr = nranks();
        std::vector<double> TL(G), TU(G);
        bool overflow = false;
        if (comm) {
            // SNP-sharded: a group's members are spread over the ranks.  T_g <= sum of the local upper bounds and
            // T_g >= every local lower bound, so the bounds of all ranks are gathered and combined
            if (gc.d_Tall.n < nT * (size_t)nr) { gc.d_Tall.alloc(nT * (size_t)nr); gc.h_Tall.alloc(nT * (size_t)nr); }
            comm_allgather_i64(comm, reinterpret_cast<const int64_t*>(gc.d_gT.p), gc.d_Tall.p, nT, s);
            IHTB_CUDA(cudaMemcpyAsync(gc.h_Tall.p, gc.d_Tall.p, nT * (size_t)nr * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
            sync();
            std::fill(TL.begin(), TL.end(), 0.0); std::fill(TU.begin(), TU.end(), 0.0);
            for (int rk = 0; rk < nr; ++rk) {
                const double* T = reinterpret_cast<const double*>(gc.h_Tall.p) + (size_t)rk * nT;
                for (size_t gi = 0; gi < G; ++gi) { TL[gi] = std::max(TL[gi], T[gi]); TU[gi] += T[G + gi]; }
                overflow = overflow || T[2 * G] != 0.0;
            }
        } else {
            IHTB_CUDA(cudaMemcpyAsync(gc.h_gT.p, gc.d_gT.p, nT * sizeof(double), cudaMemcpyDeviceToHost, s));
            sync();
            for (size_t gi = 0; gi < G; ++gi) { TL[gi] = gc.h_gT.p[gi]; TU[gi] = gc.h_gT.p[G + gi]; }
            overflow = gc.h_gT.p[2 * G] != 0.0;
        }
        IHTB_CHECK(!overflow, IHTB_ENUMERIC,
                   "degenerate group projection: too many entries of one group lie within the sweep error bound of its "
                   "2k-th largest |gradient|");
        std::vector<char> has(G, 0);
        for (int64_t j : idx) has[(size_t)gc.grp[(size_t)j]] = 1;
        std::vector<int32_t> chosen;
        std::vector<double> lows;
        for (size_t gi = 0; gi < G; ++gi) {
            if (has[gi]) chosen.push_back((int32_t)gi);
            else lows.push_back(TL[gi]);
        }
        if (gc.J > 0 && !lows.empty()) {
            // a group without support entries can reach the J best norms only if its upper bound reaches the J-th
            // largest lower bound among such groups
            const size_t need = std::min<size_t>((size_t)gc.J, lows.size());
            std::nth_element(lows.begin(), lows.begin() + (need - 1), lows.end(), std::greater<double>());
            const double thr = lows[need - 1];
            for (size_t gi = 0; gi < G; ++gi)
                if (!has[gi] && TU[gi] >= thr) chosen.push_back((int32_t)gi);
        }
        IHTB_CHECK(chosen.size() <= 65536, IHTB_ENUMERIC, "degenerate group projection: too many groups tie at the J-th norm");
        std::sort(chosen.begin(), chosen.end());
        // columns to re-score exactly: the chosen groups' lists (lcap slots each, -1 padded) + this rank's support columns
        const int nc = (int)chosen.size();
        const int64_t nsupp = (int64_t)idx.size();
        const int64_t list_slots = (int64_t)nc * gc.lcap, slots = list_slots + nsupp;
        if (slots == 0) return;
        gc.ensure_chosen(std::max(nc, 1));
        if (gc.d_oidx.n < (size_t)slots) {
            gc.d_oidx.alloc((size_t)slots); gc.d_oval.alloc((size_t)slots);
            gc.h_oidx.alloc((size_t)slots); gc.h_oval.alloc((size_t)slots);
        }
        if (nc) {
            IHTB_CUDA(cudaMemcpyAsync(gc.d_chosen.p, chosen.data(), (size_t)nc * sizeof(int32_t), cudaMemcpyHostToDevice, s));
            group_take(gc, nc, s);
        }
        std::vector<int64_t> supp_loc((size_t)nsupp);
        for (int64_t t = 0; t < nsupp; ++t) supp_loc[(size_t)t] = is_local(idx[(size_t)t]) ? idx[(size_t)t] - j0 : -1;
        upload(gc.d_oidx.p + list_slots, supp_loc.data(), (size_t)nsupp);
        xt_gather(g, gc.d_oidx.p, slots, d_r.p, 1, d_vbar.p, gc.d_oval.p, s);          // slots holding -1 are skipped
        auto take = [&](int64_t t, int64_t j, double v) {
            if (j < 0) return;
            df_exact[j] = v;
            if (t < list_slots) cand_cache.push_back(j);
        };
        if (comm) {
            const size_t blk = 2 * (size_t)slots;
            if (gc.d_blk.n < blk) gc.d_blk.alloc(blk);
            if (gc.d_blkall.n < blk * (size_t)nr) { gc.d_blkall.alloc(blk * (size_t)nr); gc.h_blkall.alloc(blk * (size_t)nr); }
            group_pack(gc.d_oidx.p, gc.d_oval.p, slots, j0, gc.d_blk.p, s);
            comm_allgather_i64(comm, gc.d_blk.p, gc.d_blkall.p, blk, s);
            IHTB_CUDA(cudaMemcpyAsync(gc.h_blkall.p, gc.d_blkall.p, blk * (size_t)nr * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
            sync();
            for (int rk = 0; rk < nr; ++rk) {
                const int64_t* b_ = gc.h_blkall.p + (size_t)rk * blk;
                for (int64_t t = 0; t < slots; ++t) {
                    double v;
                    memcpy(&v, &b_[slots + t], sizeof(double));
                    take(t, b_[t], v);
                }
            }
        } else {
            IHTB_CUDA(cudaMemcpyAsync(gc.h_oidx.p, gc.d_oidx.p, (size_t)slots * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
            IHTB_CUDA(cudaMemcpyAsync(gc.h_oval.p, gc.d_oval.p, (size_t)slots * sizeof(double), cudaMemcpyDeviceToHost, s));
            sync();
            for (int64_t t = 0; t < slots; ++t) take(t, gc.h_oidx.p[t], gc.h_oval.p[t]);
        }
        std::sort(cand_cache.begin(), cand_cache.end());
        cand_cache.erase(std::unique(cand_cache.begin(), cand_cache.end()), cand_cache.end());
        n_cand_iter += (int64_t)cand_cache.size();
    }

    // project_group_sparse! restricted to the candidate entries (position j, value v); returns the survivors
    struct GItem { double a; int64_t j; double v; int g; };
    std::vector<std::pair<int64_t, double>> project_groups(std::vector<GItem>& items) const {
        const GroupCtx& gc = *grpctx;
        std::sort(items.begin(), items.end(), [](const GItem& x, const GItem& y) { return x.a > y.a || (x.a == y.a && x.j < y.j); });
        std::unordered_map<int, std::pair<int64_t, double>> acc;       // group -> (count, norm of its k_g largest)
        for (const GItem& it : items) {
            auto& e = acc[it.g];
            if (e.first < gc.k_of(it.g, cfg.k)) { e.second += it.v * it.v; ++e.first; }
        }
        std::vector<std::pair<double, int>> order;
        for (const auto& kv : acc) order.push_back({kv.second.second, kv.first});
        std::sort(order.begin(), order.end(), [](const std::pair<double, int>& x, const std::pair<double, int>& y) {
            return x.first > y.first || (x.first == y.first && x.second < y.second);
        });
        std::unordered_map<int, int> rank;
        for (size_t i = 0; i < order.size(); ++i) rank[order[i].second] = (int)i + 1;
        std::unordered_map<int, int64_t> cnt;
        std::vector<std::pair<int64_t, double>> keep;
        for (const GItem& it : items) {
            int64_t& c_ = cnt[it.g];
            if (rank[it.g] > gc.J || c_ >= gc.k_of(it.g, cfg.k)) continue;
            ++c_;
            if (it.v != 0.0) keep.push_back({it.j, it.v});
        }
        std::sort(keep.begin(), keep.end());
        return keep;
    }

    void gradstep_group(double eta) {
        const GroupCtx& gc = *grpctx;
        std::vector<int64_t> cand = df_sparse ? dfs_idx : cand_cache;
        cand.insert(cand.end(), idx0.begin(), idx0.end());
        std::sort(cand.begin(), cand.end());
        cand.erase(std::unique(cand.begin(), cand.end()), cand.end());
        std::vector<GItem> items;
        items.reserve(cand.size());
        for (int64_t j : cand) {
            const double v = b_lookup(idx0, b0, j) + eta * df_at(j);
            items.push_back({std::fabs(v), j, v, gc.grp[(size_t)j]});
        }
        for (int64_t l = 0; l < q; ++l) c[l] = c0[l] + eta * df2[l];      // covariates are not projected (:267-269)
        auto keep = project_groups(items);
        for (int64_t l = 0; l < q; ++l) idc[l] = c[l] != 0.0;
        if (!gc.ks_vector) {                    // _choose! (src/utilities.jl:444-458) with J groups
            int64_t nonzero = (int64_t)keep.size() - zkeepn;
            for (int64_t l = 0; l < q; ++l) nonzero += idc[l] ? 1 : 0;
            const int64_t limit = (int64_t)(gc.J == 0 ? 1 : gc.J) * (cfg.k + zkeepn);
            if (nonzero > limit) {              // drop the smallest magnitudes, highest index first
                std::vector<std::pair<int64_t, double>> byabs = keep;
                std::sort(byabs.begin(), byabs.end(), [](const std::pair<int64_t, double>& x, const std::pair<int64_t, double>& y) {
                    return std::fabs(x.second) < std::fabs(y.second) || (std::fabs(x.second) == std::fabs(y.second) && x.first > y.first);
                });
                const size_t excess = std::min<size_t>((size_t)(nonzero - limit), byabs.size());
                for (size_t t = 0; t < excess; ++t)
                    keep.erase(std::find(keep.begin(), keep.end(), byabs[t]));
            }
        }
        idx.clear(); b.clear();
        for (auto& kv : keep) { idx.push_back(kv.first); b.push_back(kv.second); }
    }

    // ---- debias! (src/utilities.jl:1014-1020): b[idx] = GLM refit of y on x[:, idx]; xb / mu / df stay as they are ----
    DebiasWs debias_ws;
    void debias() {
        if (idx.empty()) return;
        std::vector<int64_t> loc(idx.size());
        for (size_t t = 0; t < idx.size(); ++t) loc[t] = is_local(idx[t]) ? idx[t] - j0 : -1;
        upload(d_cols.p, loc.data(), loc.size());
        debias_irls(g, d_y.p, cfg.dist, cfg.link, glm.nb_r, d_cols.p, (int)idx.size(), b.data(), debias_ws, s, comm);
        ++n_debias;
    }
    int64_t n_debias = 0;

    // ---- save_prev! (src/utilities.jl:702-712) ----------------------------------------------------
    double save_prev(double cur, double best) {
        idx0 = idx; b0 = b; c0 = c; idc0 = idc;
        if (cur > best) { best_idx = idx; best_b = b; best_c = c; }
        return std::max(cur, best);
    }

    // ---- check_convergence (src/utilities.jl:953-957) ---------------------------------------------
    double check_convergence() const {
        double the_norm = 0.0, b0max = 0.0;
        size_t i = 0, j = 0;
        while (i < idx.size() || j < idx0.size()) {
            double x = 0.0, y = 0.0;
            if (j >= idx0.size() || (i < idx.size() && idx[i] < idx0[j])) x = b[i++];
            else if (i >= idx.size() || idx0[j] < idx[i]) y = b0[j++];
            else { x = b[i++]; y = b0[j++]; }
            the_norm = std::max(the_norm, std::fabs(x - y));
            b0max = std::max(b0max, std::fabs(y));
        }
        for (int64_t l = 0; l < q; ++l) {
            the_norm = std::max(the_norm, std::fabs(c[l] - c0[l]));
            b0max = std::max(b0max, std::fabs(c0[l]));
        }
        return the_norm / (b0max + 1.0);
    }

    // ---- save_best_model! (src/utilities.jl:995-1006) ---------------------------------------------
    void save_best_model() {
        idx.clear(); b.clear();
        for (size_t t = 0; t < best_idx.size(); ++t)
            if (best_b[t] != 0.0) { idx.push_back(best_idx[t]); b.push_back(best_b[t]); }
        c = best_c;
        for (int64_t l = 0; l < q; ++l) idc[l] = c[l] != 0.0;
        update_xb();
        glm_update(/*add_zc=*/0);     // mu = linkinv(xb): genotype predictors only
    }

    void compute_pve() {   // var(mu) / var(y), two-pass like Statistics.var
        glm_sum2(glm, d_mu.p, d_y.p, s);
        readback_scal(2);
        double mm = h_scal.p[0] / (double)n, my = h_scal.p[1] / (double)n;
        glm_ssq2(glm, d_mu.p, mm, d_y.p, my, s);
        readback_scal(2);
        pve = h_scal.p[0] / h_scal.p[1];
    }

    // ---- init_iht_indices! (src/utilities.jl:366-438) ----------------------------------------------
    // ---- initialize_beta! + project_k! (src/utilities.jl:776-842, 412-414, 561-573): univariate regression of y on
    // [1, x_j] over the training samples for every SNP (two exact class-sum passes over the packed matrix) and covariate.
    void do_init_beta() {
        IHTB_CHECK(cfg.dist == IHTB_NORMAL, IHTB_EINVAL, "Intializing beta values only work for Gaussian phenotypes! Sorry!");
        // SNP-sharded fits: the class sums and regressions are per column (no communication); the sum of the intercepts
        // is all-reduced, and every rank's local top-k of the initial beta is all-gathered for the global projection
        DBuf<double> cls((size_t)(7 * p));           // W1 W2 Wm Y1 Y2 Ym beta
        double *W1 = cls.p, *W2 = W1 + p, *Wm = W2 + p, *Y1 = Wm + p, *Y2 = Y1 + p, *Ym = Y2 + p, *bd = Ym + p;
        init_beta_products(glm, d_xs.p, s);                                   // d_xs = w .* y
        if (geno_is_dense(g)) {            // one pass: sum w x, sum w x^2, sum w y x of every column
            dense_init_beta_moments(g, d_w.p, d_xs.p, W1, W2, Wm, s);
            n_sweeps += 1;
            init_beta_solve_moments(glm, p, W1, W2, Wm, sum_w, sum_wy, bd, s);
        } else {
            sweep_class_sums(g, d_w.p, W1, W2, Wm, s, sweep_scratch);
            sweep_class_sums(g, d_xs.p, Y1, Y2, Ym, s, sweep_scratch);
            n_sweeps += 2;
            init_beta_solve(glm, p, W1, W2, Wm, Y1, Y2, Ym, sum_w, sum_wy, g->mu.p, g->sinv.p, g->impute, bd, s);
        }                                                                     // scal[0] = sum of intercepts
        if (comm) comm_allreduce_sum_f64(comm, d_scal.p, 1, s);
        readback_scal(1);
        double c0sum = h_scal.p[0];
        // covariates 2..q (host 2x2 solves on device-reduced sums: N, sum z, sum z^2, sum z y)
        std::fill(c.begin(), c.end(), 0.0);
        if (q > 1) {
            init_beta_cov_sums(glm, s);                                         // scal[3*(l-1) + {0,1,2}]
            readback_scal(3 * ((int)q - 1));
            for (int64_t l = 1; l < q; ++l) {
                double sx = h_scal.p[3 * (l - 1)], sxx = h_scal.p[3 * (l - 1) + 1], sxy = h_scal.p[3 * (l - 1) + 2];
                double icpt = sum_wy, slope = sxy;
                double u11 = std::sqrt(sum_w), u12 = sx / u11, dd = sxx - u12 * u12;
                if (sum_w > 0 && dd > 0) {
                    double u22 = std::sqrt(dd), t1 = sum_wy / u11, t2 = (sxy - u12 * t1) / u22;
                    slope = t2 / u22; icpt = (t1 - u12 * slope) / u11;
                }
                c0sum += icpt;
                c[l] = std::min(std::max(slope, -2.0), 2.0);
            }
        }
        c[0] = std::min(std::max(c0sum / (double)(p_global + q - 1), -2.0), 2.0);
        // project_k!(v): top (k + zkeepn) of [b; c with Inf at kept covariates]
        std::vector<int64_t> cand;
        if (cfg.k > 0) {
            topk_candidates(tk, bd, nullptr, g->sinv.p, 1.0, 0.0, cfg.k, s);
            IHTB_CUDA(cudaMemcpyAsync(h_sel.p, d_sel.p, (2 + cap) * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
            sync();
            const TopkState* st = reinterpret_cast<const TopkState*>(h_sel.p);
            IHTB_CHECK(st->count <= cap, IHTB_ENUMERIC, "degenerate projection of the initial beta (too many ties)");
            cand.assign(h_sel.p + 2, h_sel.p + 2 + st->count);
            std::sort(cand.begin(), cand.end());
        }
        std::vector<double> vals(cand.size());
        if (!cand.empty()) {
            upload(d_cols.p, cand.data(), cand.size());
            take_values(bd, d_cols.p, (int64_t)cand.size(), d_gout.p, s);
            IHTB_CUDA(cudaMemcpyAsync(vals.data(), d_gout.p, cand.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
            sync();
        }
        if (comm) {        // exchange (global index, value) of the local candidates: block = [count, 0, idx[capx], bits[capx]]
            const size_t blk = 2 + 2 * (size_t)capx;
            IHTB_CHECK((int64_t)cand.size() <= capx, IHTB_ENUMERIC, "degenerate projection of the initial beta (too many ties)");
            std::vector<int64_t> mine(blk, 0);
            mine[0] = (int64_t)cand.size();
            for (size_t t = 0; t < cand.size(); ++t) {
                mine[2 + t] = cand[t] + j0;
                memcpy(&mine[2 + capx + t], &vals[t], sizeof(double));
            }
            upload(d_pack.p, mine.data(), blk);
            comm_allgather_i64(comm, d_pack.p, d_packall.p, blk, s);
            const int nr = nranks();
            IHTB_CUDA(cudaMemcpyAsync(h_packall.p, d_packall.p, nr * blk * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
            sync();
            cand.clear(); vals.clear();
            for (int rk = 0; rk < nr; ++rk) {
                const int64_t* b_ = h_packall.p + (size_t)rk * blk;
                for (int64_t t = 0; t < b_[0]; ++t) {
                    double v;
                    memcpy(&v, &b_[2 + capx + t], sizeof(double));
                    cand.push_back(b_[2 + t]);
                    vals.push_back(v);
                }
            }
        }
        struct Item { double a; int64_t pos; double v; };
        std::vector<Item> items;
        for (size_t t = 0; t < cand.size(); ++t) {
            const double w = w_at(cand[t]), a = vals[t] * w;
            items.push_back({std::fabs(a), cand[t], wt.empty() ? vals[t] : a / w});
        }
        for (int64_t l = 0; l < q; ++l)
            if (!zkeep[l]) items.push_back({std::fabs(c[l]), p_global + l, c[l]});
        std::sort(items.begin(), items.end(), [](const Item& x, const Item& y) {
            return x.a > y.a || (x.a == y.a && x.pos < y.pos);
        });
        const double thr = project_threshold(items, cfg.k);            // project_k!(v) keeps ties; no _choose! here (:412-414)
        std::vector<std::pair<int64_t, double>> keep;
        for (size_t t = 0; t < items.size(); ++t) {
            const bool kept = items[t].a >= thr;
            if (items[t].pos >= p_global) {
                if (!kept) c[items[t].pos - p_global] = 0.0;
            } else if (kept && items[t].v != 0.0) {
                keep.push_back({items[t].pos, items[t].v});
            }
        }
        std::sort(keep.begin(), keep.end());
        idx.clear(); b.clear();
        for (auto& kv : keep) { idx.push_back(kv.first); b.push_back(kv.second); }
        for (int64_t l = 0; l < q; ++l) idc[l] = c[l] != 0.0;
        // df keeps the full gradient of the intercept-only model; xb / zc / mu are NOT refreshed (:412-414)
        select_rescore(/*rerun=*/true);
    }

    void init(const uint8_t* train_mask, bool init_beta = false) {
        idx.clear(); b.clear(); idx0.clear(); b0.clear(); best_idx.clear(); best_b.clear();
        c.assign((size_t)q, 0.0); c0 = c; best_c = c; df2.assign((size_t)q, 0.0);
        idc.assign(zkeep.begin(), zkeep.end()); idc0 = idc;
        df_exact.clear(); dfs_idx.clear(); dfs_val.clear(); df_sparse = false;
        last_bt = kMaxBatch;
        d_xb.zero(s);
        const uint8_t* dm = nullptr;
        if (train_mask) {
            upload(d_mask.p, train_mask, (size_t)n);
            dm = d_mask.p;
        }
        glm_set_weights(glm, dm, s);
        readback_scal(2);
        sum_w = h_scal.p[0];
        sum_wy = h_scal.p[1];
        double ybar = h_scal.p[1] / sum_w;
        // intercept by Newton's method with the step clamped to +-1 (:394-405)
        for (int it = 0; it < 20; ++it) {
            double g1 = glm_linkinv(cfg.link, c[0]);
            double g2 = glm_mueta(cfg.link, c[0]);
            double step = (g1 - ybar) / g2;
            step = std::min(std::max(step, -1.0), 1.0);
            c[0] = c[0] - step;
            if (std::fabs(g1 - ybar) < 1e-10) break;
        }
        glm_update(1);        // zc = Z c, mu (the reference does not clamp here; xb = 0 and |c1| is small)
        init_plain = grouped() && !grpctx->ks_vector && !init_beta;
        score_and_sweep();
        init_plain = false;
        if (grouped() && grpctx->ks_vector && !init_beta) {
            // :426-430: df is projected by groups, the support is read off v.b (all zero): the fit starts from an
            // EMPTY support with the group-projected gradient, every covariate active
            std::vector<GItem> items;
            for (int64_t j : cand_cache) { double v = df_exact.at(j); items.push_back({std::fabs(v), j, v, grpctx->grp[(size_t)j]}); }
            auto keep = project_groups(items);
            for (auto& kv : keep) { dfs_idx.push_back(kv.first); dfs_val.push_back(kv.second); }
            df_sparse = true;
            idx.clear(); b.clear();
            for (int64_t l = 0; l < q; ++l) idc[l] = 1;
            inited = true;
            return;
        }
        if (init_beta) {
            do_init_beta();
            inited = true;
            return;
        }
        // first k entries chosen from the largest gradient; df itself becomes its projection (:417-425)
        std::vector<int64_t> cand = cand_cache;      // top-k of |df| with exact values (score_and_sweep)
        struct Item { double a; int64_t pos; double v; };
        std::vector<Item> items;
        for (int64_t j : cand) {
            double v = df_exact.at(j);
            const double w = w_at(j), a = v * w;
            items.push_back({std::fabs(a), j, wt.empty() ? v : a / w});
        }
        for (int64_t l = 0; l < q; ++l)
            if (!zkeep[l]) items.push_back({std::fabs(df2[l]), p_global + l, df2[l]});
        std::sort(items.begin(), items.end(), [](const Item& x, const Item& y) {
            return x.a > y.a || (x.a == y.a && x.pos < y.pos);
        });
        const double thr = project_threshold(items, cfg.k);            // ties at the k-th magnitude survive (:553-559)
        std::vector<std::pair<int64_t, double>> keep;
        for (size_t t = 0; t < items.size(); ++t) {
            const bool kept = items[t].a >= thr;
            if (items[t].pos >= p_global) {
                if (!kept) df2[items[t].pos - p_global] = 0.0;
            } else if (kept && items[t].v != 0.0) {
                keep.push_back({items[t].pos, items[t].v});
            }
        }
        std::sort(keep.begin(), keep.end());
        for (auto& kv : keep) { dfs_idx.push_back(kv.first); dfs_val.push_back(kv.second); }
        df_sparse = true;
        for (int64_t l = 0; l < q; ++l) idc[l] = zkeep[l];
        // _choose!: surplus tied entries leave the SUPPORT, the projected gradient keeps them (:450-456 zeroes v.b, which
        // is all zero here, and clears idx)
        choose_prune(keep);
        std::sort(keep.begin(), keep.end());
        idx.clear();
        for (auto& kv : keep) idx.push_back(kv.first);
        b.assign(idx.size(), 0.0);
        inited = true;
    }

    // ---- iht_one_step! (src/fit.jl:213-263) --------------------------------------------------------
    // host wall-clock per phase (seconds): stepsize, gradstep, xb + glm, score + sweep (ihtb_fit_phase_times)
    double phase[4] = {0, 0, 0, 0};
    // finer split for IHTB_CV_TIMING (multi.cu): [0] inside the sweep call (pairing wait included), [1] select_rescore,
    // [2] of that: host work after the read-back, [3] candidates re-scored, [4] init, [5] predict
    double dbg[6] = {0, 0, 0, 0, 0, 0};
    static double now() {
        return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
    }
    // The gradient step and ALL its possible backtracks in one device round trip: the candidate models
    // P_k(b0 + eta/2^s * df), s = 0..max_step, only need host work on the exact candidate values, so they are built
    // up front, evaluated together (one k_x_support over the union of their supports with an n x M output, one
    // batched k_glm_mu), and the host then walks the reference's loop `while prev_logl > logl && step < max_step`
    // over the M log-likelihoods.  Per model the arithmetic is identical to the one-at-a-time path (zero
    // coefficients add exact zeros; same blocks and reduction order), so results do not change -- only the number of
    // host<->device synchronisations per iteration (1 instead of 1 + #backtracks).
    static constexpr int kMaxBatch = 4;
    static constexpr int64_t kAdaptiveBatchN = 131072;
    int last_bt = kMaxBatch;                 // backtracks of the previous step (sizes the first batch at large n)
    DBuf<double> d_xbM, d_zcM, d_muM, d_partM, d_scalM, d_cM, d_coefM;
    HBuf<double> h_scalM;
    bool batch_ok() const {
        static const bool off = [] { const char* e = getenv("IHTB_NO_BATCH"); return e && *e == '1'; }();
        return !off && cfg.est_r == 0 && cfg.max_step >= 1 && cfg.max_step + 1 <= kMaxBatch;
    }
    struct StepModel { double eta; std::vector<int64_t> idx; std::vector<double> b, c; std::vector<uint8_t> idc; };
    std::vector<StepModel> step_models;
    void ensure_batch_buffers() {
        if (d_xbM.n < (size_t)(kMaxBatch * n)) {
            d_xbM.alloc((size_t)(kMaxBatch * n)); d_zcM.alloc((size_t)(kMaxBatch * n)); d_muM.alloc((size_t)(kMaxBatch * n));
            d_partM.alloc((size_t)kMaxBatch * GLM_MAX_BLOCKS * 3); d_scalM.alloc(kMaxBatch * 3); h_scalM.alloc(kMaxBatch * 3);
            d_cM.alloc((size_t)(kMaxBatch * q)); d_coefM.alloc((size_t)kMaxBatch * (size_t)cap);
            d_pick.alloc(1 + kMaxBatch); h_pick.alloc(1 + kMaxBatch);
        }
    }
    // host part shared by the batched and the fused step: the candidate models P_k(b0 + eta0 / 2^m df), m = 0..max_step,
    // the union of their supports, and this rank's rows of the coefficient block (uploaded)
    // models m0 .. m0 + M - 1 of the step (all of them by default): their union and coefficient block sit at offset 0 of
    // d_idx / d_coefM / d_cM, their outputs go to slots m0 .. of the n x M buffers
    struct StepPlan { int M; int m0; std::vector<int64_t> uni, loc; size_t UL; };
    StepPlan plan_step(double eta0, int m0 = 0, int m1 = -1) {
        const int Mtot = cfg.max_step + 1;
        if (m1 < 0) m1 = Mtot;
        if (m0 == 0) step_models.assign((size_t)Mtot, StepModel{});
        for (int m = m0; m < m1; ++m) {
            double e = eta0;
            for (int i = 0; i < m; ++i) e /= 2;
            if (m) { idx = idx0; b = b0; c = c0; }                       // backtrack! (src/utilities.jl:959-973)
            gradstep(e);
            step_models[(size_t)m] = StepModel{e, idx, b, c, idc};
        }
        const int M = m1 - m0;
        StepPlan pl; pl.M = M; pl.m0 = m0;
        for (int m = m0; m < m1; ++m) {
            const StepModel& md = step_models[(size_t)m];
            pl.uni.insert(pl.uni.end(), md.idx.begin(), md.idx.end());
        }
        std::sort(pl.uni.begin(), pl.uni.end());
        pl.uni.erase(std::unique(pl.uni.begin(), pl.uni.end()), pl.uni.end());
        const size_t U = pl.uni.size();
        IHTB_CHECK(U * (size_t)M <= d_coefM.n && U <= d_idx.n, IHTB_ENUMERIC, "support union too large for the batched step");
        std::vector<size_t> keep_pos;
        for (size_t t = 0; t < U; ++t)
            if (is_local(pl.uni[t])) { pl.loc.push_back(pl.uni[t] - j0); keep_pos.push_back(t); }
        pl.UL = pl.loc.size();
        std::vector<double> coefL(pl.UL * (size_t)M, 0.0), cM((size_t)(M * q));
        for (int m = 0; m < M; ++m) {
            const StepModel& md = step_models[(size_t)(m0 + m)];
            size_t u = 0;                               // both lists are sorted: one merge pass per model
            for (size_t t = 0; t < md.idx.size(); ++t) {
                if (!is_local(md.idx[t])) continue;
                const int64_t lj = md.idx[t] - j0;
                while (pl.loc[u] != lj) ++u;
                coefL[u + (size_t)m * pl.UL] = md.b[t];
            }
            for (int64_t l = 0; l < q; ++l) cM[(size_t)(m * q + l)] = md.c[(size_t)l];
        }
        if (pl.UL) {
            upload(d_idx.p, pl.loc.data(), pl.UL);
            upload(d_coefM.p, coefL.data(), coefL.size());
        }
        upload(d_cM.p, cM.data(), cM.size());
        return pl;
    }
    void adopt_model(int m) {
        const StepModel& win = step_models[(size_t)m];
        idx = win.idx; b = win.b; c = win.c; idc = win.idc;
    }
    double logl_from_sums(const double* s3) const {
        if (cfg.dist == IHTB_NORMAL) {
            const double dev = s3[0], sw = s3[2], phi = dev / (double)n, sigma = std::sqrt(phi);
            return -0.5 * (dev / phi) - sw * (0.5 * std::log(2.0 * M_PI) + std::log(sigma));
        }
        return s3[1];
    }

    void one_step_batched(double old_logl, double& eta, int& eta_step, double& new_logl) {
        ensure_batch_buffers();
        double t0 = now();
        const double eta0 = stepsize();
        double t1 = now(); phase[0] += t1 - t0;
        // Small n: all candidate models at once -- the batch costs microseconds and saves a round trip whenever the step
        // backtracks.  Long vectors (n x M products, all-reduces of n x M doubles when sharded): as many as the last step
        // needed plus one; the rest are planned and evaluated in a second round trip only if the walk in finish_batched
        // gets that far.  Per model the arithmetic does not depend on how many share a launch: same results either way.
        const int Mtot = cfg.max_step + 1;
        int first = Mtot;
        if (n >= kAdaptiveBatchN) first = std::min(Mtot, last_bt + 1 + (last_bt > 0 ? 1 : 0));
        const StepPlan pl = plan_step(eta0, 0, first);
        double t2 = now(); phase[1] += t2 - t1;
        finish_batched(pl, eta0, t2, old_logl, eta, eta_step, new_logl);
    }
    // pl covers models 0 .. pl.M - 1 of the step
    void finish_batched(const StepPlan& pl, double eta0, double t2, double old_logl, double& eta, int& eta_step,
                        double& new_logl) {
        const int Mtot = cfg.max_step + 1;
        auto eval = [&](const StepPlan& P) {                      // one device round trip for the models of plan P
            const size_t off = (size_t)P.m0 * (size_t)n;
            support_matvec_dev_m(P.UL ? d_idx.p : nullptr, (int64_t)P.UL, d_coefM.p, P.M, d_xbM.p + off);
            glm_mu_batched(glm, d_cM.p, P.M, d_xbM.p + off, d_zcM.p + off, d_muM.p + off, d_partM.p, d_scalM.p + 3 * P.m0, s);
            IHTB_CUDA(cudaMemcpyAsync(h_scalM.p + 3 * P.m0, d_scalM.p + 3 * P.m0, (size_t)(3 * P.M) * sizeof(double),
                                      cudaMemcpyDeviceToHost, s));
            sync();
        };
        int have = pl.M;
        eval(pl);
        int sidx = 0;
        new_logl = logl_from_sums(h_scalM.p);
        while (old_logl > new_logl && sidx < cfg.max_step) {                // _iht_backtrack_ (src/utilities.jl:484-486)
            ++sidx;
            if (sidx >= have) { eval(plan_step(eta0, have, Mtot)); have = Mtot; }
            new_logl = logl_from_sums(h_scalM.p + 3 * sidx);
            ++n_backtracks;
        }
        last_bt = sidx;
        adopt_model(sidx);
        eta = step_models[(size_t)sidx].eta; eta_step = sidx;
        last_dev = h_scalM.p[3 * sidx];
        const size_t nb = (size_t)n * sizeof(double);
        IHTB_CUDA(cudaMemcpyAsync(d_xb.p, d_xbM.p + (size_t)sidx * n, nb, cudaMemcpyDeviceToDevice, s));
        IHTB_CUDA(cudaMemcpyAsync(d_zc.p, d_zcM.p + (size_t)sidx * n, nb, cudaMemcpyDeviceToDevice, s));
        IHTB_CUDA(cudaMemcpyAsync(d_mu.p, d_muM.p + (size_t)sidx * n, nb, cudaMemcpyDeviceToDevice, s));
        double t3 = now(); phase[2] += t3 - t2;
        score_and_sweep();
        phase[3] += now() - t3;
        IHTB_CHECK(!std::isnan(new_logl), IHTB_ENUMERIC, "Loglikelihood function is NaN, aborting...");
        IHTB_CHECK(!std::isinf(new_logl), IHTB_ENUMERIC, "Loglikelihood function is Inf, aborting...");
    }

    // The whole iteration behind ONE host round trip: the candidate models are evaluated, the backtracking winner is
    // chosen ON THE DEVICE (k_pick_model: the reference's `while prev_logl > logl` walk over the M loglikelihoods), its
    // xb / zc / mu are adopted, and the score phase (residual, sweep, candidate selection, exact re-scoring of the
    // candidates and of the UNION of the candidate supports, next step-size denominator for the winner's support)
    // follows on the stream; the host then reads everything back at once and learns which model won.
    // Opt-in (IHTB_FUSE=1, read per step so that tests can switch it).  Measured at configs[1] on one B200: 694 vs 692
    // it/s -- the saved synchronisation (~25 us) is paid back by three more tiny kernels and the larger union gather, so
    // the default stays the two-round-trip batched step (profiles/r2_fused_step_ab.txt).
    bool fuse_ok() const {
        const char* e = getenv("IHTB_FUSE");
        return e && *e == '1' && !grouped() && denom_ready && !df_sparse;
    }
    void adopt_winner() {
        fz->winner = (int)h_pick.p[0];
        adopt_model(fz->winner);
    }
    void one_step_fused(double old_logl, double& eta, int& eta_step, double& new_logl) {
        ensure_batch_buffers();
        double t0 = now();
        const double eta0 = stepsize();                                  // host only: the denominator came back with the last sweep
        double t1 = now(); phase[0] += t1 - t0;
        const StepPlan pl = plan_step(eta0);
        const int M = pl.M;
        double t2 = now(); phase[1] += t2 - t1;
        if (comm && pl.UL > (size_t)capx / 2) {       // the union does not fit the sharded candidate block: two round trips
            finish_batched(pl, eta0, t2, old_logl, eta, eta_step, new_logl);
            return;
        }
        support_matvec_dev_m(pl.UL ? d_idx.p : nullptr, (int64_t)pl.UL, d_coefM.p, M, d_xbM.p);
        glm_mu_batched(glm, d_cM.p, M, d_xbM.p, d_zcM.p, d_muM.p, d_partM.p, d_scalM.p, s);
        glm_pick_model(glm, d_scalM.p, M, old_logl, cfg.max_step, d_pick.p, d_xbM.p, d_zcM.p, d_muM.p, s);
        FusedStep ctx;
        ctx.uni_loc = pl.loc; ctx.M = M;
        for (const StepModel& md : step_models) ctx.maxsupp = std::max(ctx.maxsupp, md.idx.size());
        double t3 = now(); phase[2] += t3 - t2;
        fz = &ctx;
        try {
            score_and_sweep();                                           // ends with the round trip and adopt_winner()
        } catch (...) {
            fz = nullptr;
            throw;
        }
        fz = nullptr;
        phase[3] += now() - t3;
        const int w = ctx.winner;
        n_backtracks += w;
        eta = step_models[(size_t)w].eta; eta_step = w;
        new_logl = h_pick.p[1 + w];
        last_dev = h_scalM.p[3 * w];
        IHTB_CHECK(!std::isnan(new_logl), IHTB_ENUMERIC, "Loglikelihood function is NaN, aborting...");
        IHTB_CHECK(!std::isinf(new_logl), IHTB_ENUMERIC, "Loglikelihood function is Inf, aborting...");
    }

    void one_step(double old_logl, double& eta, int& eta_step, double& new_logl) {
        if (batch_ok()) {
            if (fuse_ok()) one_step_fused(old_logl, eta, eta_step, new_logl);
            else one_step_batched(old_logl, eta, eta_step, new_logl);
            return;
        }
        double t0 = now();
        eta = stepsize();
        double t1 = now(); phase[0] += t1 - t0;
        gradstep(eta);
        double t2 = now(); phase[1] += t2 - t1;
        update_xb();
        new_logl = mu_r_logl();
        double t3 = now(); phase[2] += t3 - t2;
        eta_step = 0;
        while (old_logl > new_logl && eta_step < cfg.max_step) {    // _iht_backtrack_ (src/utilities.jl:484-486)
            eta /= 2;
            idx = idx0; b = b0; c = c0;                              // backtrack! (src/utilities.jl:959-973)
            double u0 = now();
            gradstep(eta);
            double u1 = now(); phase[1] += u1 - u0;
            update_xb();
            new_logl = mu_r_logl();
            phase[2] += now() - u1;
            ++eta_step;
            ++n_backtracks;
        }
        double t4 = now();
        score_and_sweep();
        phase[3] += now() - t4;
        IHTB_CHECK(!std::isnan(new_logl), IHTB_ENUMERIC, "Loglikelihood function is NaN, aborting...");
        IHTB_CHECK(!std::isinf(new_logl), IHTB_ENUMERIC, "Loglikelihood function is Inf, aborting...");
    }

    // ---- fit_iht! (src/fit.jl:145-207) -------------------------------------------------------------
    void run(ihtb_result* res, ihtb_iter_trace* trace, int64_t trace_cap) {
        IHTB_CHECK(inited, IHTB_EINVAL, "ihtb_fit_init must be called before ihtb_fit_run");
        auto t0 = std::chrono::steady_clock::now();
        int64_t launches0 = launch_counter();
        int64_t mm_iter = 0, n_steps = 0;
        double next_logl = -INFINITY, best_logl = -INFINITY;
        n_backtracks = 0;
        int64_t sweeps0 = n_sweeps;
        double sweep_ms0 = sweep_ms_total;
        for (int64_t iter = 1; iter <= cfg.max_iter; ++iter) {
            if (iter >= cfg.max_iter) {
                best_logl = save_prev(next_logl, best_logl);
                save_best_model();
                mm_iter = iter;
                break;
            }
            best_logl = save_prev(next_logl, best_logl);
            double eta; int eta_step;
            n_cand_iter = 0;
            one_step(next_logl, eta, eta_step, next_logl);
            ++n_steps;
            if (cfg.debias && iter >= 5 && idx == idx0) debias();        // src/fit.jl:187-188
            double scaled_norm = check_convergence();
            if (trace && iter - 1 < trace_cap)
                trace[iter - 1] = ihtb_iter_trace{next_logl, scaled_norm, eta, eta_step, (int32_t)n_cand_iter};
            if (iter >= cfg.min_iter && scaled_norm < cfg.tol) {
                best_logl = save_prev(next_logl, best_logl);
                save_best_model();
                mm_iter = iter;
                break;
            }
        }
        compute_pve();
        IHTB_CHECK(!p2p_failed(comm), IHTB_ECUDA, "peer-memory all-reduce timed out waiting for another rank");
        inited = false;   // like the reference, a fitted variable must be re-initialised before another fit
        if (res) {
            res->time = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
            res->logl = best_logl;
            res->iter = mm_iter;
            res->sigma_g = pve;
            res->n_sweeps = n_sweeps - sweeps0 + 1;   // + the sweep of init_iht_indices!
            res->n_backtracks = n_backtracks;
            res->sweep_seconds = (sweep_ms_total - sweep_ms0) * 1e-3;
            res->n_launches = launch_counter() - launches0;
            res->n_steps = n_steps;
        }
    }
};

extern "C" {

// Workspaces (device buffers, pinned buffers, stream, events) are expensive to create (~200 ms of cudaMalloc /
// cudaMallocHost / cudaFree at n=50k, p=500k), so destroyed fits are parked here and re-bound by the next
// ihtb_fit_create with the same shape on the same device.
static std::mutex g_cache_mu;
static std::vector<ihtb_fit*> g_cache;
static const size_t kCacheMax = 16;     // up to 8 devices x 2 shapes

static ihtb_fit* cache_take(int device, int64_t n, int64_t p, int64_t q, int cap) {
    std::lock_guard<std::mutex> lk(g_cache_mu);
    for (size_t i = 0; i < g_cache.size(); ++i) {
        ihtb_fit* f = g_cache[i];
        if (f->device == device && f->n == n && f->p == p && f->q == q && f->cap == cap) {
            g_cache.erase(g_cache.begin() + i);
            return f;
        }
    }
    return nullptr;
}

// (C linkage, internal: called by ihtb_geno_destroy)
void ihtb_internal_fit_cache_clear(int device) {
    std::vector<ihtb_fit*> drop;
    {
        std::lock_guard<std::mutex> lk(g_cache_mu);
        for (size_t i = 0; i < g_cache.size();) {
            if (device < 0 || g_cache[i]->device == device) { drop.push_back(g_cache[i]); g_cache.erase(g_cache.begin() + i); }
            else ++i;
        }
    }
    for (ihtb_fit* f : drop) { cudaSetDevice(f->device); delete f; }
}

// (C linkage, internal: multi.cu) the NEXT ihtb_fit_create of this thread gets at least this candidate capacity: paired
// cross-validation fits re-score thousands of columns per iteration
static thread_local int t_min_cap = 0;
void ihtb_internal_next_fit_min_cap(int cap) { t_min_cap = cap; }

static ihtb_fit* fit_allocate(const ihtb_geno* g, int64_t q, int cap) {
    std::unique_ptr<ihtb_fit> f(new ihtb_fit());
    int64_t n = g->n, p = g->p;
    f->device = g->device; f->n = n; f->p = p; f->q = q; f->cap = cap;
    IHTB_CUDA(cudaStreamCreateWithFlags(&f->s, cudaStreamNonBlocking));
    IHTB_CUDA(cudaEventCreate(&f->ev0));
    IHTB_CUDA(cudaEventCreate(&f->ev1));
    f->d_y.alloc(n); f->d_z.alloc(n * q); f->d_w.alloc(n); f->d_xb.alloc(n); f->d_zc.alloc(n); f->d_mu.alloc(n);
    f->d_r.alloc(n); f->d_xs.alloc(n + 2 * (size_t)cap + 64); f->d_dfa.alloc(p); f->d_mask.alloc(n);
    f->d_part.alloc((size_t)GLM_MAX_BLOCKS * (2 + q)); f->d_scal.alloc(2 + q + 8); f->d_small.alloc(2 * q);
    size_t cols_cap = 2 * (size_t)cap + 64;
    f->d_coef.alloc(cols_cap); f->d_gout.alloc(cols_cap); f->d_vbar.alloc(1);
    f->d_idx.alloc(cols_cap); f->d_cols.alloc(cols_cap);
    f->d_keyL.alloc(p); f->d_keyU.alloc(p); f->d_hist.alloc(2 * 3 * 2048); f->d_sel.alloc(2 + cap);
    f->h_scal.alloc(2 + q + 8); f->h_gout.alloc(cols_cap); f->h_sel.alloc(2 + cap);
    f->sweep_scratch = sweep_scratch_create();
    f->d_hist.zero(f->s);
    return f.release();
}

int32_t ihtb_fit_create_sharded(const ihtb_geno* g, ihtb_comm* comm, int64_t p_global, const double* y,
                                const double* z, int64_t q, const uint8_t* zkeep, const ihtb_cfg* cfg, ihtb_fit** out);

int32_t ihtb_fit_create(const ihtb_geno* g, const double* y, const double* z, int64_t q, const uint8_t* zkeep,
                        const ihtb_cfg* cfg, ihtb_fit** out) {
    return ihtb_fit_create_sharded(g, nullptr, g ? g->p : 0, y, z, q, zkeep, cfg, out);
}

int32_t ihtb_fit_create_sharded(const ihtb_geno* g, ihtb_comm* comm, int64_t p_global, const double* y,
                                const double* z, int64_t q, const uint8_t* zkeep, const ihtb_cfg* cfg, ihtb_fit** out) {
    return guard([&] {
        IHTB_CHECK(g && y && z && cfg && out, IHTB_EINVAL, "NULL argument");
        IHTB_CHECK(p_global >= g->p, IHTB_EDIM, "p_global is smaller than the local shard");
        geno_require_ready(g);
        IHTB_CHECK(!(geno_is_dense(g) && comm && comm->nranks > 1), IHTB_EUNSUPPORTED,
                   "SNP-sharded fits need PLINK handles: a dense matrix is fitted on one device");
        IHTB_CHECK(q >= 1, IHTB_EDIM, "z must have at least the intercept column");
        IHTB_CHECK(cfg->k >= 0, IHTB_EINVAL, "Value of k (max predictors per group) must be nonnegative!");
        IHTB_CHECK(cfg->max_iter >= 0, IHTB_EINVAL, "Value of max_iter must be nonnegative!");
        IHTB_CHECK(cfg->max_step >= 0, IHTB_EINVAL, "Value of max_step must be nonnegative!");
        IHTB_CHECK(cfg->tol > 2.220446049250313e-16, IHTB_EINVAL, "Value of global tol must exceed machine precision!");
        IHTB_CHECK(cfg->dist >= IHTB_NORMAL && cfg->dist <= IHTB_NEGBIN, IHTB_EINVAL, "unknown distribution");
        IHTB_CHECK(cfg->link >= IHTB_LINK_IDENTITY && cfg->link <= IHTB_LINK_INVSQ, IHTB_EINVAL, "unknown link");
        IHTB_CHECK(cfg->sweep_mode == IHTB_SWEEP_FAST || cfg->sweep_mode == IHTB_SWEEP_EXACT, IHTB_EINVAL,
                   "bad sweep_mode");
        IHTB_CHECK(cfg->k <= p_global, IHTB_EINVAL, "k cannot exceed the number of SNPs");
        IHTB_CUDA(cudaSetDevice(g->device));
        int cap = (int)std::max<int64_t>(4096, 4 * cfg->k + 1024);
        if (t_min_cap > cap) cap = t_min_cap;
        t_min_cap = 0;
        std::unique_ptr<ihtb_fit> f(cache_take(g->device, g->n, g->p, q, cap));
        if (!f) f.reset(fit_allocate(g, q, cap));
        int64_t n = g->n, p = g->p;
        f->g = g; f->cfg = *cfg;
        f->comm = (comm && comm->nranks > 1) ? comm : nullptr;
        f->j0 = f->comm ? g->j0 : 0;
        f->p_global = f->comm ? p_global : g->p;
        f->shard_j0.clear();
        if (f->comm) {
            const int nr = comm->nranks;
            // peer-memory region (collective; multi-process fits silently stay on NCCL if IPC mapping is unavailable):
            // all-reduce areas for the batched step (kMaxBatch n-vectors), gather blocks for the candidate exchange
            p2p_setup(comm, (size_t)ihtb_fit::kMaxBatch * (size_t)n,
                      (size_t)(2 + 2 * std::max<int64_t>(1024, 2 * (2 * cfg->k + 64 + 64))), f->s);
            if (f->d_selall.n < (size_t)nr * (2 + cap)) {
                f->d_selall.alloc((size_t)nr * (2 + cap));
                f->h_selall.alloc((size_t)nr * (2 + cap));
            }
            f->capx = (int)std::max<int64_t>(1024, 2 * (2 * cfg->k + 64 + 64));   // candidates | support halves
            const size_t blk = 2 + 2 * (size_t)f->capx;
            if (f->d_packall.n < (size_t)nr * blk) {
                f->d_pack.alloc(blk);
                f->d_packall.alloc((size_t)nr * blk);
                f->h_packall.alloc((size_t)nr * blk);
            }
            // exchange the shard offsets once (reuses the candidate buffers)
            int64_t mine = g->j0;
            IHTB_CUDA(cudaMemcpyAsync(f->d_sel.p, &mine, sizeof(int64_t), cudaMemcpyHostToDevice, f->s));
            comm_allgather_i64(comm, f->d_sel.p, f->d_selall.p, 1, f->s);
            f->shard_j0.resize(nr);
            IHTB_CUDA(cudaMemcpyAsync(f->shard_j0.data(), f->d_selall.p, nr * sizeof(int64_t), cudaMemcpyDeviceToHost,
                                      f->s));
            IHTB_CUDA(cudaStreamSynchronize(f->s));

        }
        f->zkeep.assign((size_t)q, 1);
        if (zkeep) for (int64_t l = 0; l < q; ++l) f->zkeep[l] = zkeep[l] ? 1 : 0;
        f->zkeepn = 0;
        for (auto v : f->zkeep) f->zkeepn += v;
        f->d_hist.zero(f->s);          // both histogram sets of the candidate selection start clean (topk.cu)
        f->inited = false; f->sweep_pending = false; f->denom_ready = false;
        f->n_sweeps = 0; f->n_backtracks = 0; f->sweep_ms_total = 0.0;
        for (int i = 0; i < 4; ++i) f->phase[i] = 0.0;
        IHTB_CHECK(cfg->est_r == 0 || cfg->dist == IHTB_NEGBIN, IHTB_EINVAL,
                   "Only negative binomial regression currently supports nuisance parameter estimation");
        IHTB_CHECK(cfg->est_r >= 0 && cfg->est_r <= 2, IHTB_EINVAL, "Only support method is Newton or MM");
        if (cfg->est_r != 0) f->h_y.assign(y, y + n); else f->h_y.clear();
        IHTB_CUDA(cudaMemcpyAsync(f->d_y.p, y, n * sizeof(double), cudaMemcpyHostToDevice, f->s));
        IHTB_CUDA(cudaMemcpyAsync(f->d_z.p, z, n * q * sizeof(double), cudaMemcpyHostToDevice, f->s));
        f->d_xb.zero(f->s); f->d_zc.zero(f->s);
        f->glm = GlmCtx{n, q, f->d_z.p, f->d_y.p, f->d_w.p, f->d_xb.p, f->d_zc.p, f->d_mu.p, f->d_r.p, f->d_part.p,
                        f->d_scal.p, cfg->dist, cfg->link, cfg->nb_r};
        if (f->d_done.n < 8) { f->d_done.alloc(8); }
        IHTB_CUDA(cudaMemsetAsync(f->d_done.p, 0, 8 * sizeof(unsigned), f->s));
        f->glm.done = f->d_done.p;                 // in-kernel finalisation of the score / glm / step-size sums (glm.cu)
        f->tk = TopkCtx{p, f->d_keyL.p, f->d_keyU.p, f->d_hist.p, reinterpret_cast<TopkState*>(f->d_sel.p),
                        f->d_sel.p + 2, f->cap};
        f->wt.clear();
        f->grpctx.reset();
        f->init_plain = false;
        f->sync();
        *out = f.release();
    });
}

int32_t ihtb_fit_set_weights(ihtb_fit* f, const double* weight) {
    return guard([&] {
        IHTB_CHECK(f, IHTB_EINVAL, "NULL fit handle");
        IHTB_CUDA(cudaSetDevice(f->g->device));
        f->set_weights(weight);
    });
}

int32_t ihtb_fit_set_groups(ihtb_fit* f, const int32_t* group, int32_t J, const int64_t* ks, int64_t n_groups) {
    return guard([&] {
        IHTB_CHECK(f, IHTB_EINVAL, "NULL fit handle");
        IHTB_CUDA(cudaSetDevice(f->g->device));
        f->set_groups(group, J, ks, n_groups);
    });
}

int32_t ihtb_fit_set_k(ihtb_fit* f, int64_t k) {
    return guard([&] {
        IHTB_CHECK(f, IHTB_EINVAL, "NULL fit handle");
        IHTB_CHECK(k >= 0 && k <= f->p, IHTB_EINVAL, "Sparsity level cannot be larger than total number of variables");
        IHTB_CHECK(4 * k + 1024 <= f->cap, IHTB_EINVAL,
                   "k exceeds the candidate capacity this fit handle was created with (create it with the largest k)");
        IHTB_CHECK(!f->grouped() || f->grpctx->ks_vector || k <= f->grpctx->kcap, IHTB_EINVAL,
                   "k exceeds the group candidate capacity (create the fit with the largest k of the path)");
        f->cfg.k = k;
    });
}

int32_t ihtb_fit_init(ihtb_fit* f, const uint8_t* train_mask) {
    return guard([&] {
        IHTB_CHECK(f, IHTB_EINVAL, "NULL fit handle");
        IHTB_CUDA(cudaSetDevice(f->g->device));
        f->init(train_mask);
    });
}

int32_t ihtb_fit_init_beta(ihtb_fit* f, const uint8_t* train_mask) {
    return guard([&] {
        IHTB_CHECK(f, IHTB_EINVAL, "NULL fit handle");
        IHTB_CUDA(cudaSetDevice(f->g->device));
        f->init(train_mask, /*init_beta=*/true);
    });
}

int32_t ihtb_fit_run(ihtb_fit* f, ihtb_result* result, ihtb_iter_trace* trace, int64_t trace_cap) {
    return guard([&] {
        IHTB_CHECK(f, IHTB_EINVAL, "NULL fit handle");
        IHTB_CUDA(cudaSetDevice(f->g->device));
        f->run(result, trace, trace_cap);
    });
}

int32_t ihtb_fit_get(const ihtb_fit* f, double* beta, double* c, double* mu, double* xb) {
    return guard([&] {
        IHTB_CHECK(f, IHTB_EINVAL, "NULL fit handle");
        IHTB_CUDA(cudaSetDevice(f->g->device));
        if (beta) {
            std::fill(beta, beta + f->p_global, 0.0);
            for (size_t t = 0; t < f->best_idx.size(); ++t) beta[f->best_idx[t]] = f->best_b[t];
        }
        if (c) std::copy(f->best_c.begin(), f->best_c.end(), c);
        if (mu) IHTB_CUDA(cudaMemcpy(mu, f->d_mu.p, f->n * sizeof(double), cudaMemcpyDeviceToHost));
        if (xb) IHTB_CUDA(cudaMemcpy(xb, f->d_xb.p, f->n * sizeof(double), cudaMemcpyDeviceToHost));
    });
}

// The model as (global column, coefficient) pairs in column order: *nnz entries exist, at most cap are written.  A caller
// holding a zeroed beta[p] (calloc) scatters them itself instead of having p doubles written (32 MB at p = 4M).
int32_t ihtb_fit_get_sparse(const ihtb_fit* f, int64_t* idx, double* val, int64_t cap, int64_t* nnz) {
    return guard([&] {
        IHTB_CHECK(f && nnz, IHTB_EINVAL, "NULL argument");
        *nnz = (int64_t)f->best_idx.size();
        for (size_t t = 0; t < f->best_idx.size() && (int64_t)t < cap; ++t) {
            if (idx) idx[t] = f->best_idx[t];
            if (val) val[t] = f->best_b[t];
        }
    });
}

int32_t ihtb_fit_predict(ihtb_fit* f, const uint8_t* test_mask, double* deviance) {
    return guard([&] {
        IHTB_CHECK(f && deviance, IHTB_EINVAL, "NULL argument");
        IHTB_CUDA(cudaSetDevice(f->g->device));
        const uint8_t* dm = nullptr;
        if (test_mask) {
            f->upload(f->d_mask.p, test_mask, (size_t)f->n);
            dm = f->d_mask.p;
        }
        glm_set_weights(f->glm, dm, f->s);     // predict! (src/cross_validation.jl:279-286)
        f->update_xb();
        f->glm_update(1);
        *deviance = f->last_dev;
    });
}

// CUDA-event stopwatch on the fit's stream (bench.py): which = 0 records the start event, 1 records the stop event
// and returns the elapsed device time between them in milliseconds.
int32_t ihtb_fit_timer(ihtb_fit* f, int32_t which, double* ms) {
    return guard([&] {
        IHTB_CHECK(f, IHTB_EINVAL, "NULL fit handle");
        IHTB_CUDA(cudaSetDevice(f->g->device));
        if (!f->tm0) { IHTB_CUDA(cudaEventCreate(&f->tm0)); IHTB_CUDA(cudaEventCreate(&f->tm1)); }
        if (which == 0) {
            IHTB_CUDA(cudaStreamSynchronize(f->s));
            IHTB_CUDA(cudaEventRecord(f->tm0, f->s));
        } else {
            IHTB_CUDA(cudaEventRecord(f->tm1, f->s));
            IHTB_CUDA(cudaEventSynchronize(f->tm1));
            float t = 0.f;
            IHTB_CUDA(cudaEventElapsedTime(&t, f->tm0, f->tm1));
            if (ms) *ms = t;
        }
    });
}

// host wall-clock seconds spent in [stepsize, gradstep, update_xb + loglikelihood, score + sweep] since creation
int32_t ihtb_fit_phase_times(const ihtb_fit* f, double* out4) {
    return guard([&] {
        IHTB_CHECK(f && out4, IHTB_EINVAL, "NULL argument");
        for (int i = 0; i < 4; ++i) out4[i] = f->phase[i];
    });
}

// (C linkage, internal: multi.cu) debug split of the score + sweep phase, see ihtb_fit::dbg
void ihtb_internal_fit_debug(const ihtb_fit* f, double* out8) {
    for (int i = 0; i < 6; ++i) out8[i] = f->dbg[i];
    out8[6] = f->sweep_ms_total * 1e-3;
    out8[7] = (double)f->n_sweeps;
}

// (C linkage, internal: multi.cu) two fits of one device share their sweeps; pairer == NULL detaches
void ihtb_internal_fit_set_pairer(ihtb_fit* f, void* pairer, int slot) {
    f->pairer = reinterpret_cast<ihtb::SweepPairer*>(pairer);
    f->pair_slot = slot;
}

int32_t ihtb_fit_destroy(ihtb_fit* f) {
    return guard([&] {
        if (!f) return;
        cudaSetDevice(f->device);
        cudaStreamSynchronize(f->s);
        f->g = nullptr;
        f->pairer = nullptr;
        {
            std::lock_guard<std::mutex> lk(g_cache_mu);
            if (g_cache.size() < kCacheMax) { g_cache.push_back(f); return; }
        }
        delete f;
    });
}

}  // extern "C"
