// One process driving several GPUs of a box (SURVEY.md 8b: `ngpu` at the drop-in boundary, so that a Julia caller of
// fit_iht / cv_iht reaches every GPU without torchrun).  A multi-device genotype handle is either
//   SHARD     : SNP columns block-partitioned over the devices -> ihtb_mfit_* runs ONE fit over all of them, one host
//               thread per device, each executing the rank code of the SNP-sharded fit (fit.cu) over an in-process
//               communicator whose collectives are peer-memory kernels (p2p.cu; no NCCL, no second process);
//   REPLICATE : the whole matrix on every device -> ihtb_mcv_run farms the (fold, k) grid of cv_iht
//               (reference src/cross_validation.jl:98-121, a `Threads.@threads` loop) over the devices from a shared
//               work queue, longest fits (largest k) first.
#include "comm.cuh"
#include "pairer.cuh"
#include <algorithm>
#include <array>
#include <atomic>
#include <chrono>
#include <functional>
#include <thread>

using namespace ihtb;

struct ihtb_mgeno {
    int mode = IHTB_MULTI_SHARD;
    int64_t n = 0, p = 0;
    std::vector<int> devices;
    std::vector<ihtb_geno*> parts;          // one per device
    std::vector<int64_t> j0, pl;            // SHARD: global offset / local columns of every part
    ~ihtb_mgeno() {
        for (size_t i = 0; i < parts.size(); ++i)
            if (parts[i]) { cudaSetDevice(devices[i]); ihtb_geno_destroy(parts[i]); }
    }
};

struct ihtb_mfit {
    const ihtb_mgeno* g = nullptr;
    std::shared_ptr<LocalGroup> group;
    std::vector<ihtb_comm*> comms;
    std::vector<ihtb_fit*> fits;
    int64_t q = 0;
};

namespace {

// run fn(rank) on one host thread per device; the first failure wins (its message becomes this thread's last error)
// and releases every rank that waits in a group barrier
int32_t on_all_ranks(int nranks, const std::vector<int>& devices, LocalGroup* group,
                     const std::function<int32_t(int)>& fn) {
    std::vector<int32_t> rc((size_t)nranks, IHTB_OK);
    std::vector<std::string> msg((size_t)nranks);
    auto body = [&](int r) {
        cudaSetDevice(devices[(size_t)r]);
        int32_t code;
        try {
            code = fn(r);
        } catch (const Error& e) {
            set_last_error(e.what());
            code = e.code;
        } catch (const std::exception& e) {
            set_last_error(e.what());
            code = IHTB_EINVAL;
        }
        rc[(size_t)r] = code;
        if (code != IHTB_OK) {
            msg[(size_t)r] = last_error();
            if (group) group->fail();
        }
    };
    std::vector<std::thread> pool;
    for (int r = 1; r < nranks; ++r) pool.emplace_back(body, r);
    body(0);
    for (auto& t : pool) t.join();
    for (int r = 0; r < nranks; ++r)
        if (rc[(size_t)r] != IHTB_OK) {
            set_last_error("device " + std::to_string(devices[(size_t)r]) + ": " + msg[(size_t)r]);
            return rc[(size_t)r];
        }
    return IHTB_OK;
}

void pick_devices(int32_t ngpu, const int32_t* devices, std::vector<int>& out) {
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) throw Error(IHTB_ECUDA, "no CUDA device available (libihtb200 has no CPU fallback)");
    IHTB_CHECK(ngpu >= 1 && ngpu <= P2P_MAX_RANKS, IHTB_EINVAL, "ngpu must be between 1 and 8");
    IHTB_CHECK(ngpu <= ndev, IHTB_EINVAL,
               "ngpu = " + std::to_string(ngpu) + " but only " + std::to_string(ndev) + " CUDA device(s) are visible");
    out.resize((size_t)ngpu);
    for (int i = 0; i < ngpu; ++i) {
        out[(size_t)i] = devices ? devices[i] : i;
        IHTB_CHECK(out[(size_t)i] >= 0 && out[(size_t)i] < ndev, IHTB_EINVAL, "device ordinal out of range");
        for (int k = 0; k < i; ++k) IHTB_CHECK(out[(size_t)k] != out[(size_t)i], IHTB_EINVAL, "a device is listed twice");
    }
}

void shard(int64_t p, int nparts, int i, int64_t* j0, int64_t* pl) {      // contiguous blocks, sizes differ by <= 1
    const int64_t base = p / nparts, rem = p % nparts;
    *j0 = i * base + std::min<int64_t>(i, rem);
    *pl = base + (i < rem ? 1 : 0);
}

ihtb_mgeno* new_mgeno(int64_t n, int64_t p, int32_t ngpu, const int32_t* devices, int32_t mode) {
    IHTB_CHECK(mode == IHTB_MULTI_SHARD || mode == IHTB_MULTI_REPLICATE, IHTB_EINVAL, "bad multi-device mode");
    std::unique_ptr<ihtb_mgeno> g(new ihtb_mgeno());
    pick_devices(ngpu, devices, g->devices);
    IHTB_CHECK(mode == IHTB_MULTI_REPLICATE || p >= ngpu, IHTB_EDIM, "fewer SNP columns than devices");
    g->mode = mode; g->n = n; g->p = p;
    g->parts.assign((size_t)ngpu, nullptr);
    g->j0.resize((size_t)ngpu); g->pl.resize((size_t)ngpu);
    for (int i = 0; i < ngpu; ++i) {
        if (mode == IHTB_MULTI_SHARD) shard(p, ngpu, i, &g->j0[(size_t)i], &g->pl[(size_t)i]);
        else { g->j0[(size_t)i] = 0; g->pl[(size_t)i] = p; }
    }
    return g.release();
}

}  // namespace

extern "C" {

int32_t ihtb_mgeno_create(const uint8_t* bed_cols, int64_t n, int64_t p, int64_t col_stride_bytes, int32_t center,
                          int32_t scale, int32_t impute, int32_t ngpu, const int32_t* devices, int32_t mode,
                          ihtb_mgeno** out) {
    int32_t rc = IHTB_OK;
    ihtb_mgeno* g = nullptr;
    rc = guard([&] {
        IHTB_CHECK(bed_cols && out, IHTB_EINVAL, "NULL argument");
        g = new_mgeno(n, p, ngpu, devices, mode);
    });
    if (rc != IHTB_OK) return rc;
    rc = on_all_ranks((int)g->devices.size(), g->devices, nullptr, [&](int r) -> int32_t {
        int32_t c = ihtb_geno_create(bed_cols + g->j0[(size_t)r] * col_stride_bytes, n, g->pl[(size_t)r], col_stride_bytes,
                                     center, scale, impute, &g->parts[(size_t)r]);
        if (c == IHTB_OK) c = ihtb_geno_set_offset(g->parts[(size_t)r], g->j0[(size_t)r]);
        return c;
    });
    if (rc != IHTB_OK) {
        std::string m = last_error();
        delete g;
        set_last_error(m);
        return rc;
    }
    *out = g;
    return IHTB_OK;
}

int32_t ihtb_mgeno_create_synthetic(int64_t n, int64_t p, uint64_t seed, double missing_rate, int32_t ngpu,
                                    const int32_t* devices, int32_t mode, ihtb_mgeno** out) {
    int32_t rc = IHTB_OK;
    ihtb_mgeno* g = nullptr;
    rc = guard([&] {
        IHTB_CHECK(out, IHTB_EINVAL, "NULL argument");
        g = new_mgeno(n, p, ngpu, devices, mode);
    });
    if (rc != IHTB_OK) return rc;
    rc = on_all_ranks((int)g->devices.size(), g->devices, nullptr, [&](int r) -> int32_t {
        return ihtb_geno_create_synthetic(n, g->pl[(size_t)r], g->j0[(size_t)r], seed, missing_rate, &g->parts[(size_t)r]);
    });
    if (rc != IHTB_OK) {
        std::string m = last_error();
        delete g;
        set_last_error(m);
        return rc;
    }
    *out = g;
    return IHTB_OK;
}

int32_t ihtb_mgeno_info(const ihtb_mgeno* g, int32_t* ngpu, int32_t* mode, int64_t* n, int64_t* p) {
    return guard([&] {
        IHTB_CHECK(g, IHTB_EINVAL, "NULL argument");
        if (ngpu) *ngpu = (int32_t)g->devices.size();
        if (mode) *mode = g->mode;
        if (n) *n = g->n;
        if (p) *p = g->p;
    });
}

int32_t ihtb_mgeno_part(const ihtb_mgeno* g, int32_t i, ihtb_geno** part, int32_t* device, int64_t* j0) {
    return guard([&] {
        IHTB_CHECK(g && i >= 0 && i < (int32_t)g->parts.size(), IHTB_EINVAL, "bad argument");
        if (part) *part = g->parts[(size_t)i];
        if (device) *device = g->devices[(size_t)i];
        if (j0) *j0 = g->j0[(size_t)i];
    });
}

int32_t ihtb_mgeno_destroy(ihtb_mgeno* g) {
    return guard([&] { delete g; });
}

// ---- one fit over a SHARD handle ---------------------------------------------------------------------------------
int32_t ihtb_mfit_destroy(ihtb_mfit* f);

int32_t ihtb_mfit_create(const ihtb_mgeno* g, const double* y, const double* z, int64_t q, const uint8_t* zkeep,
                         const ihtb_cfg* cfg, ihtb_mfit** out) {
    ihtb_mfit* f = nullptr;
    int32_t rc = guard([&] {
        IHTB_CHECK(g && y && z && cfg && out, IHTB_EINVAL, "NULL argument");
        IHTB_CHECK(g->mode == IHTB_MULTI_SHARD, IHTB_EINVAL, "ihtb_mfit needs a SHARD multi-device handle");
        f = new ihtb_mfit();
        f->g = g; f->q = q;
        const int nr = (int)g->devices.size();
        f->group = std::make_shared<LocalGroup>();
        f->group->nranks = nr;
        for (int r = 0; r < nr; ++r) f->group->devices[r] = g->devices[(size_t)r];
        f->comms.assign((size_t)nr, nullptr);
        f->fits.assign((size_t)nr, nullptr);
        for (int r = 0; r < nr; ++r) {
            ihtb_comm* c = new ihtb_comm();
            c->rank = r; c->nranks = nr; c->device = g->devices[(size_t)r];
            if (nr > 1) c->local = f->group;
            f->comms[(size_t)r] = c;
        }
    });
    if (rc != IHTB_OK) { delete f; return rc; }
    rc = on_all_ranks((int)g->devices.size(), g->devices, f->group.get(), [&](int r) -> int32_t {
        return ihtb_fit_create_sharded(g->parts[(size_t)r], f->comms[(size_t)r], g->p, y, z, q, zkeep, cfg, &f->fits[(size_t)r]);
    });
    if (rc != IHTB_OK) {
        std::string m = last_error();
        ihtb_mfit_destroy(f);
        set_last_error(m);
        return rc;
    }
    *out = f;
    return IHTB_OK;
}

#define MFIT_ALL(expr)                                                                                        \
    do {                                                                                                      \
        if (!f) { set_last_error("NULL fit handle"); return IHTB_EINVAL; }                                    \
        if (f->group->failed) { set_last_error("this multi-device fit failed earlier; destroy it"); return IHTB_ECUDA; } \
        return on_all_ranks((int)f->fits.size(), f->g->devices, f->group.get(), [&](int r) -> int32_t {        \
            ihtb_fit* fr = f->fits[(size_t)r]; (void)fr;                                                      \
            return (expr);                                                                                    \
        });                                                                                                   \
    } while (0)

int32_t ihtb_mfit_set_weights(ihtb_mfit* f, const double* weight) { MFIT_ALL(ihtb_fit_set_weights(fr, weight)); }
int32_t ihtb_mfit_set_groups(ihtb_mfit* f, const int32_t* group, int32_t J, const int64_t* ks, int64_t n_groups) {
    MFIT_ALL(ihtb_fit_set_groups(fr, group, J, ks, n_groups));
}
int32_t ihtb_mfit_set_k(ihtb_mfit* f, int64_t k) { MFIT_ALL(ihtb_fit_set_k(fr, k)); }
int32_t ihtb_mfit_init(ihtb_mfit* f, const uint8_t* train_mask, int32_t init_beta) {
    MFIT_ALL(init_beta ? ihtb_fit_init_beta(fr, train_mask) : ihtb_fit_init(fr, train_mask));
}
// every rank returns the same global model; result / trace are taken from rank 0
int32_t ihtb_mfit_run(ihtb_mfit* f, ihtb_result* result, ihtb_iter_trace* trace, int64_t trace_cap) {
    MFIT_ALL(r == 0 ? ihtb_fit_run(fr, result, trace, trace_cap) : ihtb_fit_run(fr, nullptr, nullptr, 0));
}
int32_t ihtb_mfit_predict(ihtb_mfit* f, const uint8_t* test_mask, double* deviance) {
    double dev[P2P_MAX_RANKS] = {};
    if (!f || !deviance) { set_last_error("NULL argument"); return IHTB_EINVAL; }
    int32_t rc = on_all_ranks((int)f->fits.size(), f->g->devices, f->group.get(), [&](int r) -> int32_t {
        return ihtb_fit_predict(f->fits[(size_t)r], test_mask, &dev[r]);
    });
    if (rc == IHTB_OK) *deviance = dev[0];
    return rc;
}
int32_t ihtb_mfit_get(const ihtb_mfit* f, double* beta, double* c, double* mu, double* xb) {
    if (!f) { set_last_error("NULL fit handle"); return IHTB_EINVAL; }
    cudaSetDevice(f->g->devices[0]);
    return ihtb_fit_get(f->fits[0], beta, c, mu, xb);
}
int32_t ihtb_mfit_get_sparse(const ihtb_mfit* f, int64_t* idx, double* val, int64_t cap, int64_t* nnz) {
    if (!f) { set_last_error("NULL fit handle"); return IHTB_EINVAL; }
    return ihtb_fit_get_sparse(f->fits[0], idx, val, cap, nnz);
}
// device-time stopwatch around a group of calls: which = 0 starts on every rank, 1 stops; *ms = the slowest rank
int32_t ihtb_mfit_timer(ihtb_mfit* f, int32_t which, double* ms) {
    double t[P2P_MAX_RANKS] = {};
    if (!f) { set_last_error("NULL fit handle"); return IHTB_EINVAL; }
    int32_t rc = on_all_ranks((int)f->fits.size(), f->g->devices, f->group.get(), [&](int r) -> int32_t {
        return ihtb_fit_timer(f->fits[(size_t)r], which, &t[r]);
    });
    if (rc == IHTB_OK && which == 1 && ms) *ms = *std::max_element(t, t + f->fits.size());
    return rc;
}

int32_t ihtb_mfit_destroy(ihtb_mfit* f) {
    return guard([&] {
        if (!f) return;
        for (size_t r = 0; r < f->fits.size(); ++r)
            if (f->fits[r]) { cudaSetDevice(f->g->devices[r]); ihtb_fit_destroy(f->fits[r]); }
        // the peer mappings of all ranks go away together: nobody frees a region a peer kernel could still touch
        for (size_t r = 0; r < f->comms.size(); ++r)
            if (f->comms[r]) { cudaSetDevice(f->g->devices[r]); cudaDeviceSynchronize(); }
        for (size_t r = 0; r < f->comms.size(); ++r)
            if (f->comms[r]) { cudaSetDevice(f->g->devices[r]); p2p_teardown(f->comms[r]); delete f->comms[r]; }
        delete f;
    });
}

// ---- the multivariate fit over a SHARD handle ---------------------------------------------------------------------------
struct ihtb_mmvfit {
    const ihtb_mgeno* g = nullptr;
    std::shared_ptr<LocalGroup> group;
    std::vector<ihtb_comm*> comms;
    std::vector<ihtb_mvfit*> fits;
};
int32_t ihtb_mmvfit_destroy(ihtb_mmvfit* f);

int32_t ihtb_mmvfit_create(const ihtb_mgeno* g, const double* Y, int64_t r, const double* z, int64_t q,
                           const ihtb_cfg* cfg, ihtb_mmvfit** out) {
    ihtb_mmvfit* f = nullptr;
    int32_t rc = guard([&] {
        IHTB_CHECK(g && Y && z && cfg && out, IHTB_EINVAL, "NULL argument");
        IHTB_CHECK(g->mode == IHTB_MULTI_SHARD, IHTB_EINVAL, "ihtb_mmvfit needs a SHARD multi-device handle");
        f = new ihtb_mmvfit();
        f->g = g;
        const int nr = (int)g->devices.size();
        f->group = std::make_shared<LocalGroup>();
        f->group->nranks = nr;
        for (int i = 0; i < nr; ++i) f->group->devices[i] = g->devices[(size_t)i];
        f->comms.assign((size_t)nr, nullptr);
        f->fits.assign((size_t)nr, nullptr);
        for (int i = 0; i < nr; ++i) {
            ihtb_comm* c = new ihtb_comm();
            c->rank = i; c->nranks = nr; c->device = g->devices[(size_t)i];
            if (nr > 1) c->local = f->group;
            f->comms[(size_t)i] = c;
        }
    });
    if (rc != IHTB_OK) { delete f; return rc; }
    rc = on_all_ranks((int)g->devices.size(), g->devices, f->group.get(), [&](int i) -> int32_t {
        return ihtb_mvfit_create_sharded(g->parts[(size_t)i], f->comms[(size_t)i], g->p, Y, r, z, q, cfg, &f->fits[(size_t)i]);
    });
    if (rc != IHTB_OK) {
        std::string m = last_error();
        ihtb_mmvfit_destroy(f);
        set_last_error(m);
        return rc;
    }
    *out = f;
    return IHTB_OK;
}

#define MMVFIT_ALL(expr)                                                                                       \
    do {                                                                                                       \
        if (!f) { set_last_error("NULL fit handle"); return IHTB_EINVAL; }                                     \
        if (f->group->failed) { set_last_error("this multi-device fit failed earlier; destroy it"); return IHTB_ECUDA; } \
        return on_all_ranks((int)f->fits.size(), f->g->devices, f->group.get(), [&](int i) -> int32_t {         \
            ihtb_mvfit* fr = f->fits[(size_t)i]; (void)fr;                                                     \
            return (expr);                                                                                     \
        });                                                                                                    \
    } while (0)

int32_t ihtb_mmvfit_set_k(ihtb_mmvfit* f, int64_t k) { MMVFIT_ALL(ihtb_mvfit_set_k(fr, k)); }
int32_t ihtb_mmvfit_init(ihtb_mmvfit* f, const uint8_t* train_mask, int32_t init_beta) {
    MMVFIT_ALL(init_beta ? ihtb_mvfit_init_beta(fr, train_mask) : ihtb_mvfit_init(fr, train_mask));
}
int32_t ihtb_mmvfit_run(ihtb_mmvfit* f, ihtb_result* result, ihtb_iter_trace* trace, int64_t trace_cap) {
    MMVFIT_ALL(i == 0 ? ihtb_mvfit_run(fr, result, trace, trace_cap) : ihtb_mvfit_run(fr, nullptr, nullptr, 0));
}
int32_t ihtb_mmvfit_predict(ihtb_mmvfit* f, const uint8_t* test_mask, double* mse) {
    double out[P2P_MAX_RANKS] = {};
    if (!f || !mse) { set_last_error("NULL argument"); return IHTB_EINVAL; }
    int32_t rc = on_all_ranks((int)f->fits.size(), f->g->devices, f->group.get(), [&](int i) -> int32_t {
        return ihtb_mvfit_predict(f->fits[(size_t)i], test_mask, &out[i]);
    });
    if (rc == IHTB_OK) *mse = out[0];
    return rc;
}
int32_t ihtb_mmvfit_get(const ihtb_mmvfit* f, double* beta, double* c, double* Sigma, double* sigma_g) {
    if (!f) { set_last_error("NULL fit handle"); return IHTB_EINVAL; }
    cudaSetDevice(f->g->devices[0]);
    return ihtb_mvfit_get(f->fits[0], beta, c, Sigma, sigma_g);
}
int32_t ihtb_mmvfit_destroy(ihtb_mmvfit* f) {
    return guard([&] {
        if (!f) return;
        for (size_t i = 0; i < f->fits.size(); ++i)
            if (f->fits[i]) { cudaSetDevice(f->g->devices[i]); ihtb_mvfit_destroy(f->fits[i]); }
        for (size_t i = 0; i < f->comms.size(); ++i)
            if (f->comms[i]) { cudaSetDevice(f->g->devices[i]); cudaDeviceSynchronize(); }
        for (size_t i = 0; i < f->comms.size(); ++i)
            if (f->comms[i]) { cudaSetDevice(f->g->devices[i]); p2p_teardown(f->comms[i]); delete f->comms[i]; }
        delete f;
    });
}

// ---- cv_iht: the (fold, k) grid from a shared work queue -----------------------------------------------------------------
// cv_iht (reference src/cross_validation.jl:60-131) runs q * |path| independent fits on training masks of the SAME matrix
// (allocate_fold_and_k :217-223; mu_j / sigma_j stay full-sample) and scores each on its held-out fold (predict!,
// :279-286).  The reference fans the grid out over Julia threads; here every device runs TWO fits at a time, each on its
// own host thread and stream, and their X'r sweeps are served pairwise by one pass over the matrix (pairer.cuh) -- the
// grid is bound by the sweep, so this nearly halves the matrix traffic.  Fits come from a shared atomic queue, largest
// k first (more iterations), so the devices finish together.  mses / iters are fold-major, nfolds x npath; the caller
// applies meanloss (:304-320).  IHTB_CV_PAIR=0 runs one fit at a time per device.
extern "C" void ihtb_internal_fit_set_pairer(ihtb_fit* f, void* pairer, int slot);
extern "C" void ihtb_internal_next_fit_min_cap(int cap);
extern "C" void ihtb_internal_fit_debug(const ihtb_fit* f, double* out8);

static int32_t cv_farm(const std::vector<ihtb_geno*>& parts, const std::vector<int>& devices, int64_t n, int64_t p,
                       const double* y, const double* z, int64_t q, const uint8_t* zkeep, const ihtb_cfg* cfg,
                       const int32_t* folds, int32_t nfolds, const int64_t* path, int64_t npath, const double* weight,
                       double* mses, int64_t* iters, double* busy_seconds) {
    int32_t rc = guard([&] {
        IHTB_CHECK(y && z && cfg && folds && path && mses, IHTB_EINVAL, "NULL argument");
        IHTB_CHECK(nfolds >= 1 && npath >= 1, IHTB_EINVAL, "empty cross-validation grid");
        for (int64_t t = 0; t < npath; ++t)
            IHTB_CHECK(path[t] >= 0 && path[t] <= p, IHTB_EINVAL,
                       "Sparsity level in `path` cannot be larger than total number of variables");
    });
    if (rc != IHTB_OK) return rc;
    const int64_t ngrid = (int64_t)nfolds * npath;
    std::vector<int64_t> order((size_t)ngrid);
    for (int64_t i = 0; i < ngrid; ++i) order[(size_t)i] = i;
    std::stable_sort(order.begin(), order.end(), [&](int64_t a, int64_t b) { return path[a % npath] > path[b % npath]; });
    std::atomic<int64_t> next(0);
    std::atomic<bool> stop(false);
    ihtb_cfg c = *cfg;
    c.k = *std::max_element(path, path + npath);
    const int nd = (int)devices.size();
    // Pairing pays while the PAIR sweep's looser error bound (3.1 * 2^-11 ||u||_2 sgn_j, about 0.0023 sqrt(n) null
    // standard deviations of a gradient entry) keeps the list of columns to re-score within a few thousand (they are
    // re-scored by the nibble-table gather kernel, support.cu): on by default up to n = 131072 samples (0.8 standard
    // deviations); IHTB_CV_PAIR=1 forces it (a fit whose list overflows re-sweeps alone), IHTB_CV_PAIR=0 disables it.
    const char* pe = getenv("IHTB_CV_PAIR");                  // read per call: tests switch it
    const int pair_env = pe ? atoi(pe) : -1;
    const bool want_pair = pair_env == 1 || (pair_env != 0 && n <= 131072);
    // the pair sweep needs a PLINK handle (a dense handle never pairs), FAST arithmetic and at least two fits
    const int per_dev = (want_pair && c.sweep_mode == IHTB_SWEEP_FAST && c.est_r == 0 && ngrid >= 2 &&
                         !geno_is_dense(parts[0])) ? 2 : 1;
    std::vector<std::unique_ptr<SweepPairer>> pairers((size_t)nd);
    if (per_dev == 2) {
        rc = guard([&] { for (int d = 0; d < nd; ++d) pairers[(size_t)d].reset(new SweepPairer(devices[(size_t)d])); });
        if (rc != IHTB_OK) return rc;
    }
    // est_r (NegativeBinomial nuisance parameter): the reference carries the estimate from one fit of a thread to the
    // next (v.d = mle_for_r(v), src/fit.jl:235-237; one IHTVariable per thread, src/cross_validation.jl:105), so the
    // result depends on the order of the fits.  Reproduce the single-thread order: one worker, fold-major.
    const bool sequential = c.est_r != 0;
    if (sequential) for (int64_t i = 0; i < ngrid; ++i) order[(size_t)i] = i;
    const int nworkers = sequential ? 1 : nd * per_dev;
    std::vector<int> wdev((size_t)nworkers);
    for (int w = 0; w < nworkers; ++w) wdev[(size_t)w] = devices[(size_t)(w / per_dev)];
    std::vector<double> wbusy((size_t)nworkers, 0.0);
    std::vector<std::array<double, 3>> wphase((size_t)nworkers, std::array<double, 3>{0, 0, 0});     // init, run, predict
    const bool report = getenv("IHTB_CV_TIMING") != nullptr;
    rc = on_all_ranks(nworkers, wdev, nullptr, [&](int w) -> int32_t {
        const int d = w / per_dev, slot = w % per_dev;
        SweepPairer* pr = per_dev == 2 ? pairers[(size_t)d].get() : nullptr;
        ihtb_fit* f = nullptr;
        if (pr) ihtb_internal_next_fit_min_cap(32768);       // room for the longer candidate lists of the PAIR sweep
        int32_t e = ihtb_fit_create(parts[(size_t)d], y, z, q, zkeep, &c, &f);
        if (e == IHTB_OK && weight) e = ihtb_fit_set_weights(f, weight);
        if (e == IHTB_OK && pr) ihtb_internal_fit_set_pairer(f, pr, slot);
        std::vector<uint8_t> train((size_t)n), test((size_t)n);
        int last_fold = -1;
        const auto t0 = std::chrono::steady_clock::now();
        while (e == IHTB_OK && !stop.load()) {
            const int64_t pos = next.fetch_add(1);
            if (pos >= ngrid) break;
            const int64_t i = order[(size_t)pos];
            const int fold = (int)(i / npath) + 1;
            const int64_t t = i % npath;
            if (fold != last_fold) {
                for (int64_t s = 0; s < n; ++s) { test[(size_t)s] = folds[s] == fold; train[(size_t)s] = !test[(size_t)s]; }
                last_fold = fold;
            }
            ihtb_result res;
            double dev = 0.0;
            e = ihtb_fit_set_k(f, path[t]);
            const auto ta = std::chrono::steady_clock::now();
            if (e == IHTB_OK) e = ihtb_fit_init(f, train.data());
            const auto tb = std::chrono::steady_clock::now();
            if (e == IHTB_OK) e = ihtb_fit_run(f, &res, nullptr, 0);
            const auto tc = std::chrono::steady_clock::now();
            if (e == IHTB_OK) e = ihtb_fit_predict(f, test.data(), &dev);
            const auto td = std::chrono::steady_clock::now();
            wphase[(size_t)w][0] += std::chrono::duration<double>(tb - ta).count();
            wphase[(size_t)w][1] += std::chrono::duration<double>(tc - tb).count();
            wphase[(size_t)w][2] += std::chrono::duration<double>(td - tc).count();
            if (e == IHTB_OK) {
                mses[i] = dev;
                if (iters) iters[i] = res.iter;
            }
        }
        wbusy[(size_t)w] = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        if (report && f) {
            double ph[4] = {0, 0, 0, 0}, dg[8] = {0};
            ihtb_fit_phase_times(f, ph);
            ihtb_internal_fit_debug(f, dg);
            fprintf(stderr, "[cv worker %d] busy %.3f s: init %.3f run %.3f predict %.3f | run phases: stepsize %.3f gradstep %.3f "
                    "xb+glm %.3f score+sweep %.3f | sweep call (incl. pairing wait) %.3f, select+rescore %.3f (host part %.3f), "
                    "sweep kernels %.3f s over %.0f sweeps, %.0f candidates re-scored; pair sweeps %lld solo %lld\n",
                    w, wbusy[(size_t)w], wphase[(size_t)w][0], wphase[(size_t)w][1], wphase[(size_t)w][2], ph[0], ph[1], ph[2],
                    ph[3], dg[0], dg[1], dg[2], dg[6], dg[7], dg[3], pr ? (long long)pr->n_pair : 0LL,
                    pr ? (long long)pr->n_solo : 0LL);
        }
        if (pr) pr->leave();                          // the partner sweeps alone from now on (also on an error)
        if (e != IHTB_OK) {
            stop.store(true);
            std::string m = last_error();
            if (f) { ihtb_internal_fit_set_pairer(f, nullptr, 0); ihtb_fit_destroy(f); }
            set_last_error(m);
            return e;
        }
        ihtb_internal_fit_set_pairer(f, nullptr, 0);
        return ihtb_fit_destroy(f);
    });
    if (busy_seconds)
        for (int d = 0; d < nd; ++d) {
            double b = 0.0;
            for (int sl = 0; sl < per_dev; ++sl) b = std::max(b, wbusy[(size_t)(d * per_dev + sl)]);
            busy_seconds[d] = b;
        }
    return rc;
}

// cv_iht in one call on ONE device
int32_t ihtb_cv_run(const ihtb_geno* g, const double* y, const double* z, int64_t q, const uint8_t* zkeep,
                    const ihtb_cfg* cfg, const int32_t* folds, int32_t nfolds, const int64_t* path, int64_t npath,
                    const double* weight, double* mses, int64_t* iters) {
    if (!g) { set_last_error("NULL argument"); return IHTB_EINVAL; }
    std::vector<ihtb_geno*> parts{const_cast<ihtb_geno*>(g)};
    std::vector<int> devices{g->device};
    return cv_farm(parts, devices, g->n, g->p, y, z, q, zkeep, cfg, folds, nfolds, path, npath, weight, mses, iters, nullptr);
}

// ... and over the replicas of a REPLICATE handle; busy_seconds[ngpu] (optional) = wall time every device spent fitting
int32_t ihtb_mcv_run(const ihtb_mgeno* g, const double* y, const double* z, int64_t q, const uint8_t* zkeep,
                     const ihtb_cfg* cfg, const int32_t* folds, int32_t nfolds, const int64_t* path, int64_t npath,
                     const double* weight, double* mses, int64_t* iters, double* busy_seconds) {
    if (!g) { set_last_error("NULL argument"); return IHTB_EINVAL; }
    if (g->mode != IHTB_MULTI_REPLICATE) {
        set_last_error("ihtb_mcv_run needs a REPLICATE multi-device handle");
        return IHTB_EINVAL;
    }
    return cv_farm(g->parts, g->devices, g->n, g->p, y, z, q, zkeep, cfg, folds, nfolds, path, npath, weight, mses, iters,
                   busy_seconds);
}

}  // extern "C"
