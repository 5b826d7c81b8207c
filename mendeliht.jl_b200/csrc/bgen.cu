// BGEN 1.2 (layout 2) ingest: the inflated probability block of a variant -> one column of a dense handle.
//
// A BGEN layout-2 block stores each probability as a B-bit integer v meaning v / (2^B - 1), so the dosage of a
// biallelic diploid sample is exactly an integer code / D with D = 2^B - 1:
//   unphased (a = P(11), b = P(12), c = D - a - b):  code = b + 2 c             (copies of the second allele)
//   phased (h = P(haplotype carries allele 1)):      code = 2 D - h1 - h2
//   first allele:                                    2 D - code
// k_bgen_decode turns the raw blocks into those codes on the device and writes them straight into the padded columns:
// FIX16 handles store the code (the handle's denominator must be D, so B <= 15 and code <= 65534), Float64 handles
// store code / D by one IEEE FP64 division (any B <= 32).  A missing sample becomes IHTB_DOSAGE16_MISSING or NaN, as
// from_dosages / from_array encode it, so the handle needs standardize = 1 exactly when the file has missing samples.
// Everything after the load (finalize, decode, stats, sweeps, fits) is the dense.cu code path unchanged.
//
// Validation is deterministic: every failing CTA (one variant) posts key = column << 36 | reason << 32 | aux with
// atomicMin, so the error reported is that of the lowest failing column (lowest reason, then lowest sample), whatever
// the launch order.
//
// Sample selection (ihtb_geno_select_bgen_samples): row i of the handle is file sample rows[i].  The row map is the
// ROWMAP template flag of k_bgen_decode, so a load without a selection runs the kernel it always ran.  A block then holds
// n_file samples; only the kept ones are read and checked, and errors name file sample indices (< 2^32, the aux field).
#include "common.cuh"
#include <atomic>
#include <algorithm>
#include <string.h>
#include <thread>

namespace ihtb {

constexpr int BG_THREADS = 256;
constexpr int64_t BG_PAD = 16;                 // zero bytes after the staged data: the last 64-bit window stays in bounds
constexpr int64_t BG_MAX_COLS = int64_t(1) << 27;   // columns per call: the column field of the error key is 28 bits
static std::atomic<int64_t> g_bgen_batch_bytes{int64_t(64) << 20};

// why a block was rejected; the order is the order of the checks (and of the error reported for one column)
enum BgenReason : uint32_t {
    BG_SHORT_HEADER = 1,     // IHTB_EINVAL       block shorter than its header
    BG_N = 2,                // IHTB_EDIM         N != the handle's n, or n_file of a selection (aux = N)
    BG_K = 3,                // IHTB_EUNSUPPORTED K != 2 (aux = K)
    BG_PHASED = 4,           // IHTB_EINVAL       phased flag not 0 / 1 (aux = flag)
    BG_BITS = 5,             // IHTB_EINVAL       B = 0 or B > 32 (aux = B)
    BG_DEN = 6,              // IHTB_EINVAL       FIX16 handle and 2^B - 1 != denominator (aux = B)
    BG_SHORT_DATA = 7,       // IHTB_EINVAL       block shorter than header + ceil(2 N B / 8)
    BG_PLOIDY = 8,           // IHTB_EUNSUPPORTED non-missing kept sample with ploidy != 2 (aux = file sample)
    BG_SUM = 9,              // IHTB_EDOMAIN      unphased a + b > 2^B - 1 (aux = file sample)
};

struct BgenTarget {
    uint8_t* x;              // the handle's columns (uint16 codes or FP64 values)
    int64_t ld, n;
    uint64_t n_file;         // samples per block: n, or the n_file of a selection
    const uint32_t* rows;    // ROWMAP: row i is file sample rows[i] (ld entries, zero after n)
    int fix16;
    int allele;              // 1 or 2: the allele whose copies are counted
    uint64_t den;            // FIX16: the handle's denominator
};

// the 8 bytes at base + byte, from the two aligned 64-bit words that hold them (base is 16-byte aligned and the staged
// data is followed by BG_PAD bytes, so w[1] is in bounds for every byte of the data)
__device__ __forceinline__ uint64_t bg_window(const uint8_t* __restrict__ base, uint64_t byte) {
    const uint64_t* w = reinterpret_cast<const uint64_t*>(base) + (byte >> 3);
    const uint32_t sh = (uint32_t)(byte & 7) * 8;
    return (__ldg(w) >> sh) | ((__ldg(w + 1) << 1) << (63 - sh));   // sh = 0: the second term is 0
}
// the B-bit value at bit `bit` (least-significant bit first); B <= 32, so bit & 7 + B <= 39 bits of one window
__device__ __forceinline__ uint64_t bg_value(const uint8_t* __restrict__ base, uint64_t bit, uint64_t mask) {
    return (bg_window(base, bit >> 3) >> (bit & 7)) & mask;
}

// grid = ncols (one CTA per variant).  Block c is base[off[c] .. off[c + 1]) and becomes column j0 + c; c_call is the
// index of block 0 within the caller's call (the column field of the error key).  ROWMAP: row i reads file sample
// t.rows[i]; otherwise row i is file sample i.
template <bool ROWMAP>
__global__ void __launch_bounds__(BG_THREADS)
k_bgen_decode(const uint8_t* __restrict__ base, const int64_t* __restrict__ off, BgenTarget t, int64_t j0,
              int64_t c_call, unsigned long long* __restrict__ err) {
    const int64_t c = blockIdx.x;
    const uint64_t b0 = (uint64_t)off[c], len = (uint64_t)(off[c + 1] - off[c]);
    const unsigned long long key0 = (unsigned long long)(c_call + c) << 36;
    // header: every thread reads the same bytes, so the control flow below is block-uniform
    uint32_t reason = 0, aux = 0;
    uint64_t N = 0, B = 0, phased = 0;
    if (len < 8) {
        reason = BG_SHORT_HEADER;
    } else {
        const uint64_t h = bg_window(base, b0);
        N = h & 0xffffffffu;
        const uint32_t K = (uint32_t)(h >> 32) & 0xffffu;
        if (N != t.n_file) { reason = BG_N; aux = (uint32_t)N; }
        else if (K != 2) { reason = BG_K; aux = K; }
        else if (len < 10 + N) reason = BG_SHORT_HEADER;
        else {
            const uint64_t h2 = bg_window(base, b0 + 8 + N);
            phased = h2 & 0xff;
            B = (h2 >> 8) & 0xff;
            if (phased > 1) { reason = BG_PHASED; aux = (uint32_t)phased; }
            else if (B == 0 || B > 32) { reason = BG_BITS; aux = (uint32_t)B; }
            else if (t.fix16 && (1ull << B) - 1 != t.den) { reason = BG_DEN; aux = (uint32_t)B; }
            else if (len < 10 + N + (2 * N * B + 7) / 8) reason = BG_SHORT_DATA;
        }
    }
    if (reason) {
        if (threadIdx.x == 0) atomicMin(err, key0 | (unsigned long long)reason << 32 | aux);
        return;
    }
    const uint64_t D = (1ull << B) - 1;
    const uint64_t pl = b0 + 8, dbit = (b0 + 10 + N) * 8;
    const int64_t n = t.n, ld = t.ld;
    unsigned long long bad = ~0ull;                // this thread's lowest (reason << 32 | file sample)
    // code of file sample i (i < N): false when the sample is missing (or rejected, recorded in `bad`)
    auto code_of = [&](uint64_t i, uint64_t& code) -> bool {
        const uint32_t pb = base[pl + i];
        if (pb & 0x80) return false;
        if ((pb & 63) != 2) {
            bad = min(bad, (unsigned long long)BG_PLOIDY << 32 | (uint64_t)i);
            return false;
        }
        const uint64_t q = dbit + 2 * i * B;
        const uint64_t v0 = bg_value(base, q, D), v1 = bg_value(base, q + B, D);
        uint64_t c2;                                 // copies of the second allele, in units of 1 / D
        if (phased) {
            c2 = 2 * D - v0 - v1;
        } else {
            if (v0 + v1 > D) {
                bad = min(bad, (unsigned long long)BG_SUM << 32 | i);
                return false;
            }
            c2 = v1 + 2 * (D - v0 - v1);
        }
        code = t.allele == 2 ? c2 : 2 * D - c2;
        return true;
    };
    if (t.fix16) {                                 // 8 rows per thread, one 16-byte store (ld is a multiple of 256)
        uint16_t* col = reinterpret_cast<uint16_t*>(t.x) + (j0 + c) * ld;
        for (int64_t i0 = (int64_t)threadIdx.x * 8; i0 < ld; i0 += BG_THREADS * 8) {
            uint32_t w[4] = {0u, 0u, 0u, 0u};
            uint32_t fi[8];                            // file sample of each row
            if (ROWMAP) {
                const uint4 r0 = __ldg(reinterpret_cast<const uint4*>(t.rows + i0));
                const uint4 r1 = __ldg(reinterpret_cast<const uint4*>(t.rows + i0) + 1);
                fi[0] = r0.x; fi[1] = r0.y; fi[2] = r0.z; fi[3] = r0.w;
                fi[4] = r1.x; fi[5] = r1.y; fi[6] = r1.z; fi[7] = r1.w;
            }
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const int64_t i = i0 + e;
                uint64_t code = 0;
                uint32_t v = 0;                        // rows n..ld-1 stay zero
                if (i < n) v = code_of(ROWMAP ? (uint64_t)fi[e] : (uint64_t)i, code) ? (uint32_t)code
                                                                                       : (uint32_t)IHTB_DOSAGE16_MISSING;
                w[e >> 1] |= v << (16 * (e & 1));
            }
            *reinterpret_cast<uint4*>(col + i0) = make_uint4(w[0], w[1], w[2], w[3]);
        }
    } else {                                       // 2 rows per thread, one 16-byte store (ld is a multiple of 128)
        double* col = reinterpret_cast<double*>(t.x) + (j0 + c) * ld;
        const double dd = (double)D;
        for (int64_t i0 = (int64_t)threadIdx.x * 2; i0 < ld; i0 += BG_THREADS * 2) {
            double v[2];
            uint32_t fi[2];
            if (ROWMAP) {
                const uint2 r = __ldg(reinterpret_cast<const uint2*>(t.rows + i0));
                fi[0] = r.x; fi[1] = r.y;
            }
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int64_t i = i0 + e;
                uint64_t code = 0;
                v[e] = 0.0;
                if (i < n) v[e] = code_of(ROWMAP ? (uint64_t)fi[e] : (uint64_t)i, code)
                                      ? __ddiv_rn((double)code, dd) : __longlong_as_double(0x7ff8000000000000ll);
            }
            *reinterpret_cast<double2*>(col + i0) = make_double2(v[0], v[1]);
        }
    }
    if (bad != ~0ull) atomicMin(err, key0 | bad);
}

static void bgen_throw(unsigned long long key, int64_t j_first, int32_t den, int64_t n_file, bool selected) {
    const int64_t c = (int64_t)(key >> 36);
    const uint32_t reason = (uint32_t)(key >> 32) & 15u, aux = (uint32_t)key;
    const std::string where = "BGEN block " + std::to_string(c) + " (column " + std::to_string(j_first + c) + "): ";
    switch (reason) {
        case BG_SHORT_HEADER: throw Error(IHTB_EINVAL, where + "the block is shorter than its header");
        case BG_N: throw Error(IHTB_EDIM, where + "the block holds N = " + std::to_string(aux) + " samples, " +
                                              (selected ? "the sample selection's n_file = " + std::to_string(n_file)
                                                        : std::string("the handle n differs")));
        case BG_K: throw Error(IHTB_EUNSUPPORTED, where + std::to_string(aux) + " alleles (only biallelic variants)");
        case BG_PHASED: throw Error(IHTB_EINVAL, where + "phased flag " + std::to_string(aux) + " is not 0 or 1");
        case BG_BITS: throw Error(IHTB_EINVAL, where + "B = " + std::to_string(aux) + " bits per probability (1..32)");
        case BG_DEN: throw Error(IHTB_EINVAL, where + "B = " + std::to_string(aux) + " bits, but the handle's denominator " +
                                                  std::to_string(den) + " is not 2^B - 1");
        case BG_SHORT_DATA: throw Error(IHTB_EINVAL, where + "the block is shorter than its header + ceil(2 N B / 8) bytes");
        case BG_PLOIDY: throw Error(IHTB_EUNSUPPORTED, where + (selected ? "file sample " : "sample ") + std::to_string(aux) +
                                                           " is not diploid (only diploid samples)");
        case BG_SUM: throw Error(IHTB_EDOMAIN, where + (selected ? "file sample " : "sample ") + std::to_string(aux) +
                                                   ": P(11) + P(12) exceeds 1 (a + b > 2^B - 1)");
        default: throw Error(IHTB_EINVAL, where + "rejected");
    }
}

// Two pinned staging buffers with a device twin and a stream each, the error word, and the sample selection.  Kept on
// the handle between calls (g->bgen_stage, released at finalize): a file arrives in many ~64 MB calls, and pinning
// 2 x 64 MB of host memory costs far more than copying it.
struct BgenStage {
    static constexpr int NB = 2;
    size_t cap = 0;
    bool loaded = false;                 // a load call has run: the selection is fixed from here on
    int64_t n_file = 0;                  // > 0: a selection is set, and every block holds n_file samples
    DBuf<uint32_t> rows;                 // the selection's row map, ld entries (zero after n: vector loads stay in bounds)
    HBuf<uint8_t> hbuf[NB];
    DBuf<uint8_t> dbuf[NB];
    DBuf<unsigned long long> err;
    cudaStream_t st[NB] = {nullptr, nullptr};
    cudaEvent_t done[NB] = {nullptr, nullptr};
    void sync() {
        for (int i = 0; i < NB; ++i) if (st[i]) cudaStreamSynchronize(st[i]);
    }
    ~BgenStage() {
        sync();
        for (int i = 0; i < NB; ++i) {
            if (st[i]) cudaStreamDestroy(st[i]);
            if (done[i]) cudaEventDestroy(done[i]);
        }
    }
};

static BgenStage& bgen_stage(ihtb_geno* g, size_t cap = 0) {
    auto* s = static_cast<BgenStage*>(g->bgen_stage.get());
    if (!s) {
        s = new BgenStage();
        g->bgen_stage.reset(s, [](void* q) { delete static_cast<BgenStage*>(q); });
        for (int i = 0; i < BgenStage::NB; ++i) {
            IHTB_CUDA(cudaStreamCreateWithFlags(&s->st[i], cudaStreamNonBlocking));
            IHTB_CUDA(cudaEventCreateWithFlags(&s->done[i], cudaEventDisableTiming));
        }
        s->err.alloc(1);
    }
    if (s->cap < cap) {                                // grow with headroom: batches of later calls vary in size
        s->sync();
        const size_t want = cap + cap / 4;
        s->cap = 0;
        for (int i = 0; i < BgenStage::NB; ++i) {
            s->hbuf[i].alloc(want);
            s->dbuf[i].alloc(want);
        }
        s->cap = want;
    }
    return *s;
}

// Host -> HBM: the blocks go in batches of about g_bgen_batch_bytes (whole blocks, at least one) through the two
// staging buffers: the host threads copy batch i + 1 into one while the other's cudaMemcpyAsync and decode of batch i
// run on its stream.  A staged batch is [relative offsets][data][BG_PAD zero bytes].
static void bgen_load(ihtb_geno* g, const uint8_t* blocks, const int64_t* offsets, int64_t j_first, int64_t ncols,
                      int allele) {
    const int64_t limit = std::max<int64_t>(1, g_bgen_batch_bytes.load());
    std::vector<int64_t> cut{0};
    int64_t max_bytes = 0, max_cols = 0;
    for (int64_t c = 0; c < ncols;) {
        int64_t e = c + 1;
        while (e < ncols && offsets[e + 1] - offsets[c] <= limit) ++e;
        max_bytes = std::max(max_bytes, offsets[e] - offsets[c]);
        max_cols = std::max(max_cols, e - c);
        cut.push_back(e);
        c = e;
    }
    const int64_t doff = ceil_div((max_cols + 1) * 8, 16) * 16;
    BgenStage& s = bgen_stage(g, (size_t)(doff + ceil_div(max_bytes, 16) * 16 + BG_PAD));
    s.loaded = true;
    const bool sel = s.n_file > 0;
    unsigned nt = std::thread::hardware_concurrency();
    nt = std::max(1u, std::min(nt, 16u));
    BgenTarget t{g->dense.p, g->ld, g->n, (uint64_t)(sel ? s.n_file : g->n), sel ? s.rows.p : nullptr,
                 g->dtype == IHTB_DENSE_FIX16 ? 1 : 0, allele, (uint64_t)g->den};
    try {
        IHTB_CUDA(cudaMemsetAsync(s.err.p, 0xff, sizeof(unsigned long long), s.st[0]));
        IHTB_CUDA(cudaStreamSynchronize(s.st[0]));
        for (size_t k = 0; k + 1 < cut.size(); ++k) {
            const int b = (int)(k & 1);
            const int64_t c0 = cut[k], c1 = cut[k + 1], h = c1 - c0;
            const int64_t bytes = offsets[c1] - offsets[c0];
            IHTB_CUDA(cudaEventSynchronize(s.done[b]));        // the buffer's previous batch is decoded
            uint8_t* hb = s.hbuf[b].p;
            int64_t* ro = reinterpret_cast<int64_t*>(hb);
            for (int64_t c = 0; c <= h; ++c) ro[c] = offsets[c0 + c] - offsets[c0];
            uint8_t* dst = hb + doff;
            const uint8_t* src = blocks + offsets[c0];
            const unsigned use = (unsigned)std::max<int64_t>(1, std::min<int64_t>(nt, bytes >> 20));
            auto copy = [=](unsigned ti) {
                const int64_t a = bytes * ti / use, e = bytes * (ti + 1) / use;
                memcpy(dst + a, src + a, (size_t)(e - a));
            };
            std::vector<std::thread> pool;
            for (unsigned ti = 1; ti < use; ++ti) pool.emplace_back(copy, ti);
            copy(0);
            for (auto& th : pool) th.join();
            memset(dst + bytes, 0, (size_t)BG_PAD);
            IHTB_CUDA(cudaMemcpyAsync(s.dbuf[b].p, hb, (size_t)(doff + bytes + BG_PAD), cudaMemcpyHostToDevice, s.st[b]));
            if (sel)
                IHTB_LAUNCH(k_bgen_decode<true>, (unsigned)h, BG_THREADS, 0, s.st[b], s.dbuf[b].p + doff,
                            reinterpret_cast<const int64_t*>(s.dbuf[b].p), t, j_first + c0, c0, s.err.p);
            else
                IHTB_LAUNCH(k_bgen_decode<false>, (unsigned)h, BG_THREADS, 0, s.st[b], s.dbuf[b].p + doff,
                            reinterpret_cast<const int64_t*>(s.dbuf[b].p), t, j_first + c0, c0, s.err.p);
            IHTB_CUDA(cudaEventRecord(s.done[b], s.st[b]));
        }
        for (int i = 0; i < BgenStage::NB; ++i) IHTB_CUDA(cudaStreamSynchronize(s.st[i]));
    } catch (...) {
        s.sync();
        throw;
    }
    unsigned long long key = 0;
    IHTB_CUDA(cudaMemcpy(&key, s.err.p, sizeof(key), cudaMemcpyDeviceToHost));
    if (key != ~0ull) bgen_throw(key, j_first, g->den, s.n_file, sel);
}

}  // namespace ihtb

using namespace ihtb;

extern "C" {

int32_t ihtb_geno_load_bgen_columns(ihtb_geno* g, const uint8_t* blocks, const int64_t* offsets, int64_t j_first,
                                    int64_t ncols, int32_t allele) {
    return guard([&] {
        IHTB_CHECK(g && offsets, IHTB_EINVAL, "NULL argument");
        IHTB_CHECK(geno_is_dense(g), IHTB_EINVAL, "not a dense handle (BGEN dosages load into dense handles)");
        IHTB_CHECK(!g->ready, IHTB_EINVAL, "handle is already finalized");
        IHTB_CHECK(g->dtype == IHTB_DENSE_FIX16 || g->dtype == IHTB_DENSE_F64, IHTB_EINVAL,
                   "BGEN dosages load into IHTB_DENSE_FIX16 or IHTB_DENSE_F64 handles");
        IHTB_CHECK(allele == 1 || allele == 2, IHTB_EINVAL, "allele must be 1 or 2");
        IHTB_CHECK(j_first >= 0 && ncols >= 0 && j_first + ncols <= g->p, IHTB_EDIM, "column range outside the matrix");
        IHTB_CHECK(ncols <= BG_MAX_COLS, IHTB_EINVAL, "at most 2^27 blocks per call");
        if (ncols == 0) return;
        IHTB_CHECK(blocks || offsets[ncols] == offsets[0], IHTB_EINVAL, "NULL argument");
        IHTB_CHECK(offsets[0] >= 0, IHTB_EINVAL, "offsets[0] must be >= 0");
        for (int64_t c = 0; c < ncols; ++c)
            IHTB_CHECK(offsets[c + 1] >= offsets[c], IHTB_EINVAL,
                       "offsets must be non-decreasing (offsets[" + std::to_string(c + 1) + "] < offsets[" +
                           std::to_string(c) + "])");
        IHTB_CUDA(cudaSetDevice(g->device));
        bgen_load(g, blocks, offsets, j_first, ncols, allele);
    });
}

int32_t ihtb_geno_select_bgen_samples(ihtb_geno* g, const int64_t* rows, int64_t n_file) {
    return guard([&] {
        IHTB_CHECK(g && rows, IHTB_EINVAL, "NULL argument");
        IHTB_CHECK(geno_is_dense(g), IHTB_EINVAL, "not a dense handle (BGEN dosages load into dense handles)");
        IHTB_CHECK(!g->ready, IHTB_EINVAL, "handle is already finalized");
        IHTB_CHECK(g->dtype == IHTB_DENSE_FIX16 || g->dtype == IHTB_DENSE_F64, IHTB_EINVAL,
                   "BGEN dosages load into IHTB_DENSE_FIX16 or IHTB_DENSE_F64 handles");
        const auto* st = static_cast<const BgenStage*>(g->bgen_stage.get());
        IHTB_CHECK(!(st && st->loaded), IHTB_EINVAL,
                   "BGEN columns are already loaded: select the samples before the first ihtb_geno_load_bgen_columns");
        const int64_t n = g->n;
        IHTB_CHECK(n <= n_file && n_file <= (int64_t)UINT32_MAX, IHTB_EINVAL,
                   "n_file = " + std::to_string(n_file) + " must lie in [n = " + std::to_string(n) + ", 2^32 - 1]");
        for (int64_t i = 0; i < n; ++i)
            IHTB_CHECK(rows[i] >= 0 && rows[i] < n_file, IHTB_EINVAL,
                       "rows[" + std::to_string(i) + "] = " + std::to_string(rows[i]) + " is outside [0, n_file = " +
                           std::to_string(n_file) + ")");
        // a repeat: sort (row, position) and report the pair whose later position is lowest
        std::vector<std::pair<int64_t, int64_t>> sorted((size_t)n);
        for (int64_t i = 0; i < n; ++i) sorted[(size_t)i] = {rows[i], i};
        std::sort(sorted.begin(), sorted.end());
        int64_t first = -1, second = -1;
        for (size_t k = 1; k < sorted.size(); ++k)
            if (sorted[k].first == sorted[k - 1].first && (k < 2 || sorted[k - 2].first != sorted[k].first) &&
                (second < 0 || sorted[k].second < second)) {
                first = sorted[k - 1].second;
                second = sorted[k].second;
            }
        IHTB_CHECK(second < 0, IHTB_EINVAL,
                   "rows[" + std::to_string(first) + "] and rows[" + std::to_string(second) + "] are both file sample " +
                       std::to_string(rows[second]));
        IHTB_CUDA(cudaSetDevice(g->device));
        std::vector<uint32_t> map((size_t)g->ld, 0u);
        for (int64_t i = 0; i < n; ++i) map[(size_t)i] = (uint32_t)rows[i];
        BgenStage& s = bgen_stage(g);
        s.n_file = 0;
        s.rows.alloc(map.size());
        IHTB_CUDA(cudaMemcpyAsync(s.rows.p, map.data(), map.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, s.st[0]));
        IHTB_CUDA(cudaStreamSynchronize(s.st[0]));
        s.n_file = n_file;
    });
}

int32_t ihtb_bgen_set_batch_bytes(int64_t bytes) {
    g_bgen_batch_bytes.store(bytes > 0 ? bytes : int64_t(64) << 20);
    return IHTB_OK;
}

}  // extern "C"
