// EXACT X'v sweep for sm_100a: FP64 lookup tables indexed by NIBBLE (2 genotypes), same TMA pipeline as sweep_lut.cu.
//
// A shift/compare/select/DFMA per genotype (the first exact kernel) is issue-bound at 0.6 TB/s.  A byte-indexed FP64
// table like the FAST kernel's would need 256 KB per 512-sample slab, so here a table row covers 2 samples: for the 32
// words w of a column chunk and the 8 nibbles t of a word
//     T[t][value][w] = dosage(value & 3) * u[512*slab + 16*w + 2*t] + dosage(value >> 2) * u[512*slab + 16*w + 2*t + 1],
// u = v - mean(v) in FP64: 8 * 16 * 32 doubles = 32 KB.  Lane w owns word w of a column chunk; the 32 lanes of one
// LDS.64 read 32 consecutive doubles of a row whatever the data are (2 wavefronts, the minimum for 256 bytes).  Rows
// are 256 bytes apart inside a 4 KB-aligned table per nibble position, so the address is base | ((word >> 4t) & 15) << 8:
// one shift and one LOP3 per lookup.  Per packed word and column: 8 LDS.64 + 8 DADD instead of 16 x (shift, compare,
// select, DFMA).  Producer warp, stage ring, per-group "full" barriers, butterfly reduction and the [slab][column]
// partial-sum layout (FP64 here) are those of sweep_lut.cu; the epilogue adds the slabs in order.  Deterministic.
#include "common.cuh"

namespace ihtb {

namespace {

constexpr int X_STAGE_COLS = 128;
constexpr int X_STAGE_BYTES = X_STAGE_COLS * 128;
constexpr int X_STAGES = 8;
constexpr int X_TABLE_BYTES = 8 * 16 * 32 * 8;                  // 32 KB
constexpr int X_CW = 16, X_G = 2;                                // consumer warps, groups
constexpr int X_SMEM_BYTES = 4096 + 4096 + X_TABLE_BYTES + X_STAGES * X_STAGE_BYTES;   // barriers + alignment slack + table + ring

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n"
        "W_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@!p bra W_%=;\n\t}"
        ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ double lds_f64(uint32_t addr) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts_f64(uint32_t addr, double v) {
    asm volatile("st.shared.f64 [%0], %1;" ::"r"(addr), "d"(v) : "memory");
}
__device__ __forceinline__ void consumer_bar() {
    asm volatile("bar.sync 1, %0;" ::"n"(X_CW * 32) : "memory");
}

// 512 consumer threads: thread -> (nibble t, word w) pair and one half of the 16 values
// cls selects what a 2-bit code contributes: 0 = the additive dosage (0, 0, 1, 2 for codes 00, 01, 10, 11; the X'v
// sweep), 1 = the heterozygote indicator (code 10), 2 = the homozygote indicator (code 11) -- the class sums
// sum_i v_i [g_ij = 1] and sum_i v_i [g_ij = 2] that initialize_beta! needs (src/utilities.jl:776-812)
__device__ __forceinline__ void build64(uint32_t tab, const double* __restrict__ v, double vbar, int64_t n,
                                        int64_t slab, int tid, int cls) {
    const int pair = tid & 255, half = tid >> 8;
    const int t = pair >> 5, w = pair & 31;
    const int64_t i0 = slab * 512 + 16 * w + 2 * t;
    const double u0 = (i0 < n) ? __dsub_rn(v[i0], vbar) : 0.0;
    const double u1 = (i0 + 1 < n) ? __dsub_rn(v[i0 + 1], vbar) : 0.0;
    const uint32_t base = tab + (uint32_t)t * 4096u + 8u * (uint32_t)w;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        const int val = half * 8 + e;
        const int c0 = val & 3, c1 = val >> 2;
        double a0, a1;
        if (cls == 0) {
            a0 = (c0 == 2) ? u0 : ((c0 == 3) ? __dadd_rn(u0, u0) : 0.0);
            a1 = (c1 == 2) ? u1 : ((c1 == 3) ? __dadd_rn(u1, u1) : 0.0);
        } else {
            const int hit = cls == 1 ? 2 : 3;
            a0 = (c0 == hit) ? u0 : 0.0;
            a1 = (c1 == hit) ? u1 : 0.0;
        }
        sts_f64(base + (uint32_t)val * 256u, __dadd_rn(a0, a1));
    }
}

__device__ __forceinline__ uint4 lds_u128(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}

// Quad-interleaved tiles (common.cuh): a stage holds 32 quads of 512 bytes, 16 bytes per (quad, word), so one LDS.128
// per lane fetches word `lane` of four columns (same wavefront count as four LDS.32).
// p is the number of columns stored per slab (p4); p_out the number of result columns.
__global__ void __launch_bounds__((X_CW + 1) * 32, 1)
k_sweep_lut64(const uint8_t* __restrict__ bed, int64_t cs_s, int64_t p, int64_t p_out, int64_t n, int64_t n_slabs,
              const double* __restrict__ v, const double* __restrict__ vbar_p, double* __restrict__ part, int cls) {
    const double vbar = vbar_p ? *vbar_p : 0.0;         // class sums are taken of the vector itself
    constexpr int WPG = X_CW / X_G;                 // warps per group
    constexpr int CPW = X_STAGE_COLS / WPG;         // columns per warp per unit (16)
    constexpr int S = X_STAGES;
    constexpr int period = (S % X_G == 0) ? S : S * X_G;
    extern __shared__ __align__(128) uint8_t smem_raw[];
    const uint32_t base = smem_u32(smem_raw);
    const uint32_t bar_full = (base + 127u) & ~127u;            // full[g*S + st], then empty[st]
    const uint32_t bar_empty = bar_full + 8u * X_G * S;
    const uint32_t tab = (bar_empty + 8u * S + 4095u) & ~4095u;
    const uint32_t stage0 = tab + X_TABLE_BYTES;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    const int64_t n_cblocks = (p + X_STAGE_COLS - 1) / X_STAGE_COLS;
    const int64_t units = n_slabs * n_cblocks;
    const int64_t u_beg = units * (int64_t)blockIdx.x / gridDim.x;
    const int64_t u_end = units * (int64_t)(blockIdx.x + 1) / gridDim.x;
    if (u_beg >= u_end) return;
    const int64_t slab_beg = u_beg / n_cblocks, slab_end = (u_end - 1) / n_cblocks;   // inclusive
    const int ncb = (int)n_cblocks;

    if (threadIdx.x == 0) {
        for (int s = 0; s < S; ++s) {
            for (int g = 0; g < X_G; ++g) mbar_init(bar_full + 8u * (g * S + s), 1);
            mbar_init(bar_empty + 8u * s, WPG);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (warp == X_CW) {
        // ===== producer warp: one contiguous 16 KB bulk copy per (slab, column block) unit =====
        int st = 0; uint32_t ph = 0;
        int grp_of = 0;
        for (int64_t slab = slab_beg; slab <= slab_end; ++slab) {
            const int cb0 = (slab == slab_beg) ? (int)(u_beg - slab * n_cblocks) : 0;
            const int cb1 = (slab == slab_end) ? (int)(u_end - slab * n_cblocks) : ncb;
            for (int cb = cb0; cb < cb1; ++cb) {
                const int64_t j0 = (int64_t)cb * X_STAGE_COLS;
                const int ncols = (int)((p - j0 < X_STAGE_COLS) ? (p - j0) : X_STAGE_COLS);
                const uint32_t fullbar = bar_full + 8u * (uint32_t)(grp_of * S + st);
                mbar_wait(bar_empty + 8u * st, ph ^ 1u);
                if (lane == 0) {
                    mbar_expect_tx(fullbar, (uint32_t)ncols * 128u);
                    bulk_g2s(stage0 + (uint32_t)st * X_STAGE_BYTES, bed + j0 * 128 + slab * cs_s, (uint32_t)ncols * 128u, fullbar);
                }
                if (++st == S) { st = 0; ph ^= 1u; }
                if (++grp_of == X_G) grp_of = 0;
            }
        }
    } else {
        // ===== consumer warps =====
        const int tid = threadIdx.x;
        const int grp = warp / WPG, wg = warp % WPG;
        uint32_t lb[8];
#pragma unroll
        for (int t = 0; t < 8; ++t) lb[t] = tab + (uint32_t)t * 4096u + 8u * (uint32_t)lane;
        constexpr int LPC = 32 / CPW;
        const int col = wg * CPW + lane / LPC;
        const bool writer = (lane & (LPC - 1)) == 0;
        const uint32_t lane_off = (uint32_t)(wg * CPW) * 128u + 16u * (uint32_t)lane;
        int st = grp % S, ip = grp % period; uint32_t ph = (uint32_t)((grp / period) & 1);
        const uint32_t my_full = bar_full + 8u * (uint32_t)(grp * S);
        int i_next = grp;
        int i_base = 0;
        for (int64_t slab = slab_beg; slab <= slab_end; ++slab) {
            const int cb0 = (slab == slab_beg) ? (int)(u_beg - slab * n_cblocks) : 0;
            const int cb1 = (slab == slab_end) ? (int)(u_end - slab * n_cblocks) : ncb;
            consumer_bar();
            build64(tab, v, vbar, n, slab, tid, cls);
            consumer_bar();
            double* __restrict__ outp = part + slab * p_out + col;
            const int i_end = i_base + (cb1 - cb0);
            for (; i_next < i_end; i_next += X_G) {
                const int cb = cb0 + (i_next - i_base);
                mbar_wait(my_full + 8u * st, ph);
                const uint32_t colbase = stage0 + (uint32_t)st * X_STAGE_BYTES + lane_off;
                double acc[CPW];
                uint4 q4 = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
                for (int c = 0; c < CPW; ++c) {
                    if ((c & 3) == 0) q4 = lds_u128(colbase + 512u * (c >> 2));
                    const uint32_t w = (c & 3) == 0 ? q4.x : (c & 3) == 1 ? q4.y : (c & 3) == 2 ? q4.z : q4.w;
                    const double d0 = lds_f64(lb[0] | ((w << 8) & 0xF00u));
                    const double d1 = lds_f64(lb[1] | ((w << 4) & 0xF00u));
                    const double d2 = lds_f64(lb[2] | (w & 0xF00u));
                    const double d3 = lds_f64(lb[3] | ((w >> 4) & 0xF00u));
                    const double d4 = lds_f64(lb[4] | ((w >> 8) & 0xF00u));
                    const double d5 = lds_f64(lb[5] | ((w >> 12) & 0xF00u));
                    const double d6 = lds_f64(lb[6] | ((w >> 16) & 0xF00u));
                    const double d7 = lds_f64(lb[7] | ((w >> 20) & 0xF00u));
                    acc[c] = __dadd_rn(__dadd_rn(__dadd_rn(d0, d1), __dadd_rn(d2, d3)),
                                       __dadd_rn(__dadd_rn(d4, d5), __dadd_rn(d6, d7)));
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_empty + 8u * st);
                int o = 16;
#pragma unroll
                for (int h = CPW / 2; h >= 1; h >>= 1, o >>= 1) {
                    const bool upper = (lane & o) != 0;
#pragma unroll
                    for (int c = 0; c < h; ++c) {
                        const double send = upper ? acc[c] : acc[c + h];
                        const double keep = upper ? acc[c + h] : acc[c];
                        acc[c] = __dadd_rn(keep, __shfl_xor_sync(0xffffffffu, send, o));
                    }
                }
#pragma unroll
                for (int oo = 16 / CPW; oo >= 1; oo >>= 1) acc[0] = __dadd_rn(acc[0], __shfl_xor_sync(0xffffffffu, acc[0], oo));
                const int jj = cb * X_STAGE_COLS + col;
                if (writer && jj < (int)p_out) outp[cb * X_STAGE_COLS] = acc[0];
                st += X_G; if (st >= S) st -= S;
                ip += X_G; if (ip >= period) { ip -= period; ph ^= 1u; }
            }
            i_base = i_end;
        }
    }
}

}  // namespace

// d_part is [stride/128][p] doubles
void sweep_exact_lut_partials(const ihtb_geno* g, const double* d_v, const double* d_vbar, double* d_part, cudaStream_t s,
                              int cls) {
    IHTB_CHECK(g->p < (int64_t(1) << 31) - 256, IHTB_EDIM, "more than 2^31 SNP columns on one GPU");
    const int64_t n_slabs = g->stride / 128;
    const int64_t units = n_slabs * ceil_div(g->p4, X_STAGE_COLS);
    int grid = g->sm_count;
    if (units < grid) grid = (int)units;
    ensure_dynamic_smem(k_sweep_lut64, X_SMEM_BYTES);
    IHTB_LAUNCH(k_sweep_lut64, grid, (X_CW + 1) * 32, X_SMEM_BYTES, s, g->bed.p, g->cs_s, g->p4, g->p, g->n, n_slabs, d_v,
                d_vbar, d_part, cls);
}

}  // namespace ihtb
