// FAST X'v sweep for sm_100a: byte-indexed lookup tables ("four Russians") in shared memory.
//
// Why: at 6.5 TB/s a B200 SM must consume ~100 genotypes per clock; a decode + FMA per genotype is ALU-bound at
// less than half of that (SURVEY.md App. D).  Here every packed byte (4 genotypes) costs one PRMT (address),
// one conflict-free LDS.32 (table lookup) and one FADD.
//
// Work decomposition: the matrix is cut into slabs of 512 samples (= one 128-byte chunk per column).  A CTA owns a
// contiguous range of (slab, 128-column block) units.  For its current slab it builds, from u = v - mean(v) (FP32),
//     T[t][value][w] = sum_{s<4} dosage((value >> 2s) & 3) * u[512*slab + 16*w + 4*t + s]
// for the 32 words w of a chunk and the 4 bytes t of a word: 4*256*32 floats = 128 KB.  The 32 lanes of an LDS always
// look up 32 different word positions w, so they hit 32 distinct banks whatever the data bytes are.
// The 256 rows (value) of a table are 256 bytes apart and each pair of tables fills one 64 KB-aligned window of
// shared memory, so the lookup address is a single PRMT: byte 1 of a per-lane base register is replaced by the
// data byte.
//
// Data movement: a producer warp streams column chunks into a ring of 16 KB shared-memory stages with
// cp.async.bulk (TMA bulk copy, SASS UBLKCP) completing on mbarriers; 16 consumer warps take them in groups.
// On the ternary copy, FAST sweep (the default): lane l owns one column and walks its 32 words, so the column sum
// is a register tree and each 128-byte chunk costs 5 shared-memory data-pipe passes (4 lookups, 1 read-back).
// Otherwise lane w owns word w of 16 columns, which a butterfly of shuffles (a sixth pass) reduces across the warp.
// Both orders add the same word sums in the same pairwise tree.  Slab partial sums are written as FP32
// [slab][column]; the epilogue (sweep.cu) adds them in FP64 in slab order.  Everything is deterministic.
#include "lut_common.cuh"
#include <stdlib.h>

namespace ihtb {

constexpr int LUT_STAGE_COLS = 128;
constexpr int LUT_STAGE_BYTES = LUT_STAGE_COLS * 128;
constexpr int LUT_MAX_STAGES = 8;
constexpr int LUT_MAX_GROUPS = 4;
constexpr uint32_t LUT_BAR_BYTES = 8u * (LUT_MAX_GROUPS + 1) * LUT_MAX_STAGES;
constexpr int LUT_SMEM_BYTES = 232448;   // 227 KB: everything the SM has

// shared-memory plan (computed identically by every thread)
struct LutPlan {
    uint32_t bar_full, bar_empty;      // arrays of 8-byte mbarriers
    uint32_t tab;                      // 64 KB-aligned, 128 KB
    uint32_t lo0, hi0;                 // first stage below / above the tables (512-byte aligned)
    int n_lo, n_stages;
    __device__ __forceinline__ uint32_t stage(int s) const {
        return (s < n_lo) ? lo0 + (uint32_t)s * LUT_STAGE_BYTES : hi0 + (uint32_t)(s - n_lo) * LUT_STAGE_BYTES;
    }
};
__device__ __forceinline__ LutPlan lut_plan(uint32_t base, uint32_t bytes) {
    LutPlan pl;
    uint32_t end = base + bytes;
    pl.tab = (base + 65535u) & ~65535u;
    pl.bar_full = 0; pl.bar_empty = 0; pl.n_stages = 0;
    uint32_t lo = (base + 127u) & ~127u, lo_end = pl.tab;
    uint32_t hi = pl.tab + LUT_TABLE_BYTES, hi_end = end;
    // barriers at the first free spot: full[LUT_MAX_GROUPS][LUT_MAX_STAGES] then empty[LUT_MAX_STAGES]
    if (lo + LUT_BAR_BYTES <= lo_end) { pl.bar_full = lo; lo += LUT_BAR_BYTES; }
    else { pl.bar_full = hi; hi += LUT_BAR_BYTES; }
    pl.bar_empty = pl.bar_full + 8u * LUT_MAX_GROUPS * LUT_MAX_STAGES;
    // stages start at multiples of 512 bytes: the one-column-per-lane consumer XORs word offsets into address bits 2..8
    lo = (lo + 511u) & ~511u; hi = (hi + 511u) & ~511u;
    pl.lo0 = lo; pl.hi0 = hi;
    pl.n_lo = (lo_end > lo) ? (int)((lo_end - lo) / LUT_STAGE_BYTES) : 0;
    if (pl.n_lo > LUT_MAX_STAGES) pl.n_lo = LUT_MAX_STAGES;
    int n_hi = (hi_end > hi) ? (int)((hi_end - hi) / LUT_STAGE_BYTES) : 0;
    pl.n_stages = pl.n_lo + n_hi;
    if (pl.n_stages > LUT_MAX_STAGES) pl.n_stages = LUT_MAX_STAGES;
    return pl;
}

// Units: u = slab * n_cblocks + cblock, CTA b handles [u_begin(b), u_begin(b+1)), slab by slab.
// CW consumer warps in G groups (+ 1 producer warp).  Group g consumes the CTA's units with (local index % G) == g, and
// each of its CW/G warps reduces CPW = 128*G/CW columns of that unit, so per-unit bookkeeping is amortised over 16
// columns per warp while 16 warps keep the shared-memory pipe busy.
// The groups share one ring of S stages (unit i uses stage i % S) and one "empty" mbarrier per stage, but every
// group has its OWN "full" mbarrier per stage: the producer signals full[i % G][i % S].  A warp must observe every
// phase of a barrier it waits on -- a parity wait issued a whole phase early is satisfied by the preceding phase
// (the mbarrier ABA hazard) and the warp would read a slot before it is refilled.  With per-group full barriers a
// group sees exactly the fills meant for it, in order, while the groups still progress independently.
//
// QUAD: quad-interleaved tiles (common.cuh): a stage is 32 quads of 512 bytes, one LDS.128 per lane fetches word
//       `lane` of four columns (same wavefronts as four LDS.32, a quarter of the instructions).  `p` is then the padded
//       column count stored per slab and p_out the number of result columns.
// H2:   the PAIR sweep -- two right-hand sides per pass.  The table entries are half2 (v0 | v1), so ONE lookup serves
//       both: per word four half2 lookups added with HADD2, converted to FP32 and reduced across lanes in FP32.
//       Entries are scaled by a power of two per right-hand side (max |u| <= 2^9: entries <= 2^12, sums of four
//       <= 2^14, no overflow); part is [2][n_slabs][p_out] floats of the SCALED sums.  Error bound, per column sum:
//       one FP16 rounding per table entry + two levels of HADD2 on partial sums bounded by twice the absolute sum of
//       the 16 samples of a word: 3 * 2^-11 * 2 ||u||_1 < 2^-8 ||u||_1 (FP32 and subnormal terms are below 1e-5 of that).
// TERN: the stream is the handle's ternary copy (common.cuh): five dosages per byte, 640 samples per chunk.  Bytes are
//       opaque table keys to this kernel, so only the table builders differ.
// COL:  TERN && !H2 (the default FAST sweep): 4 groups of 4 warps, 32 columns per warp, and each lane walks the 32 words
//       of ONE column, so its column sum ends in registers and there is no butterfly.  Shared-memory data-pipe
//       wavefronts per 128-byte chunk: 4 lookups + 1 read-back, against 6 with the shuffles.  See the consumer below.
template <int CW, int G, bool QUAD, bool H2, bool TERN>
__global__ void __launch_bounds__((CW + 1) * 32, 1)
k_sweep_lut(const uint8_t* __restrict__ bed, int64_t cs_j, int64_t cs_s, int64_t p, int64_t p_out, int64_t n,
            int64_t n_slabs, const double* __restrict__ v, const double* __restrict__ v1,
            const double* __restrict__ vbar_p, const float* __restrict__ scale_p, float* __restrict__ part,
            uint32_t dyn_bytes) {
    const double vbar = vbar_p[0];
    const double vbar1 = H2 ? vbar_p[1] : 0.0;
    const float sc0 = H2 ? scale_p[0] : 1.0f, sc1 = H2 ? scale_p[1] : 1.0f;
    constexpr bool COL = TERN && !H2;                // one column per lane
    constexpr int WPG = CW / G;                      // warps per group
    constexpr int CPW = LUT_STAGE_COLS / WPG;        // columns per warp per unit
    static_assert(G <= LUT_MAX_GROUPS, "barrier block holds LUT_MAX_GROUPS full barriers per stage");
    static_assert(!QUAD || CPW % 4 == 0, "quad layout: a warp owns whole quads");
    static_assert(!H2 || (CW == 16 && CPW == 16), "pair sweep: 512 table builders, 16 columns per warp");
    static_assert(!TERN || (QUAD && CW == 16), "ternary tiles: quad layout, 512 table builders");
    static_assert(!COL || CPW == 32, "one column per lane: 32 columns per warp");
    extern __shared__ __align__(128) uint8_t smem_raw[];
    const LutPlan pl = lut_plan(smem_u32(smem_raw), dyn_bytes);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int S = pl.n_stages;
    // (group, stage) pairs repeat with period lcm(S, G) in the unit index
    int period = S;
    while (period % G != 0) period += S;

    const int64_t n_cblocks = (p + LUT_STAGE_COLS - 1) / LUT_STAGE_COLS;
    const int64_t units = n_slabs * n_cblocks;
    const int64_t u_beg = units * (int64_t)blockIdx.x / gridDim.x;
    const int64_t u_end = units * (int64_t)(blockIdx.x + 1) / gridDim.x;
    if (u_beg >= u_end) return;
    const int64_t slab_beg = u_beg / n_cblocks, slab_end = (u_end - 1) / n_cblocks;   // inclusive
    const int ncb = (int)n_cblocks;

    if (threadIdx.x == 0) {
        for (int s = 0; s < S; ++s) {
            for (int g = 0; g < G; ++g) mbar_init(pl.bar_full + 8u * (g * LUT_MAX_STAGES + s), 1);
            mbar_init(pl.bar_empty + 8u * s, WPG);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (warp == CW) {
        // ===== producer warp: stream column chunks with bulk async copies =====
        int st = 0; uint32_t ph = 0;                 // stage of the next unit, parity of its "empty" phase
        int grp_of = 0;                              // group that owns the next unit (local unit index % G)
        for (int64_t slab = slab_beg; slab <= slab_end; ++slab) {
            const int cb0 = (slab == slab_beg) ? (int)(u_beg - slab * n_cblocks) : 0;
            const int cb1 = (slab == slab_end) ? (int)(u_end - slab * n_cblocks) : ncb;    // exclusive
            for (int cb = cb0; cb < cb1; ++cb) {
                const int64_t j0 = (int64_t)cb * LUT_STAGE_COLS;
                const int ncols = (int)((p - j0 < LUT_STAGE_COLS) ? (p - j0) : LUT_STAGE_COLS);
                const uint32_t fullbar = pl.bar_full + 8u * (uint32_t)(grp_of * LUT_MAX_STAGES + st);
                mbar_wait(pl.bar_empty + 8u * st, ph ^ 1u);
                const uint8_t* src = bed + j0 * cs_j + slab * cs_s;
                if (cs_j == 128) {               // slab-major tiles (plain or quad-interleaved): one contiguous copy
                    if (lane == 0) {
                        mbar_expect_tx(fullbar, (uint32_t)ncols * 128u);
                        bulk_g2s(pl.stage(st), src, (uint32_t)ncols * 128u, fullbar);
                    }
                } else {                          // column-major layout: one 128-byte copy per column
                    if (lane == 0) mbar_expect_tx(fullbar, (uint32_t)ncols * 128u);
                    __syncwarp();
                    for (int c = lane; c < ncols; c += 32)
                        bulk_g2s(pl.stage(st) + 128u * c, src + (int64_t)c * cs_j, 128u, fullbar);
                }
                if (++st == S) { st = 0; ph ^= 1u; }
                if (++grp_of == G) grp_of = 0;
            }
        }
    } else {
        // ===== consumer warps =====
        const int tid = threadIdx.x;      // 0 .. CW*32-1
        const int grp = warp / WPG, wg = warp % WPG;
        // per-lane base registers for the 4 bytes of a word: byte 1 gets replaced by the data byte
        uint32_t lb[4];
#pragma unroll
        for (int t = 0; t < 4; ++t)
            lb[t] = pl.tab + (uint32_t)(t >> 1) * 65536u + (uint32_t)(t & 1) * 128u + 4u * (uint32_t)lane;
        constexpr int NACC = H2 ? 2 * CPW : CPW;      // values reduced per warp and unit
        constexpr int LPC = 32 / NACC > 0 ? 32 / NACC : 1;   // lanes holding the same value after the butterfly
        // after the butterfly lane l holds value index l / LPC: (rhs, column) = (idx / CPW, idx % CPW)
        // TERN (PAIR; the FAST sweep takes the COL path): accumulator slot c of lane l holds value c ^ (l & (NACC - 1)) --
        // the ternary tiles store component i of the quad word w as column i ^ (w & 3) (geno.cu), the lane reads quad
        // q ^ ((l >> 2) & 3), and the pair tables of word positions >= 16 carry the right-hand sides in swapped halves -- so
        // every butterfly level is "keep the low half, add the partner's high half": no selects (2 per value otherwise:
        // 18 % of the PAIR kernel's instructions, which was issue-bound).  Lane l ends with value l & (NACC - 1).
        // COL: NACC = 32 and every lane writes column l of the warp (vidx = l).
        const int vidx = TERN ? (lane & (NACC - 1)) : lane / LPC;
        const int col = wg * CPW + vidx % CPW;        // column (within a unit) this lane stores
        const bool writer = TERN ? (lane < NACC) : (lane & (LPC - 1)) == 0;
        const uint32_t lqs = TERN ? ((((uint32_t)lane >> 2) & 3u) << 9) : 0u;
        const uint32_t lane_off = (uint32_t)(wg * CPW) * 128u + (QUAD ? 16u : 4u) * (uint32_t)lane;
        // COL: lane l owns component ci = l & 3 of the warp's quad ql = l >> 2, i.e. column 4 ql + ci = l of the warp, and
        // at step s = 0..31 takes word position w = w0 ^ s, w0 = 8 ci + ql.  In the tiles that word sits at byte
        // 512 ql + 16 w + 4 (ci ^ (w & 3)) = D0 ^ K(s) with K(s) = 16 s + 4 (s & 3) (disjoint bit fields), so with
        // 512-byte aligned stages its address is one XOR with a constant.  Per step the 32 lanes read 32 distinct banks,
        // 4 (w & 7) + (ci ^ (w & 3)), and their table lookups (bank w) too.
        const uint32_t w0 = 8u * ((uint32_t)lane & 3u) + ((uint32_t)lane >> 2);
        const uint32_t col_off = (uint32_t)(wg * CPW) * 128u + ((uint32_t)lane >> 2) * 512u + 16u * w0 +
                                 4u * (((uint32_t)lane & 3u) ^ (w0 & 3u));
        // lookup base Y = [4 w | 128 + 4 w | window of t = 0, 1 | window of t = 2, 3]; step s uses Y0 ^ (4 s * 0x0101) and
        // byte t of the word needs address [Y.b(t & 1) | data byte t | Y.b(2 + (t >> 1)) | 0]: one PRMT (the zero is the
        // sign of a window byte, which is < 0x80)
        const uint32_t y0 = 4u * w0 | (128u + 4u * w0) << 8 | (pl.tab >> 16) << 16 | ((pl.tab >> 16) + 1u) << 24;
        // this group consumes local unit indices i = grp, grp+G, ...: stage i % S, full-barrier parity (i / period) & 1
        int st = grp % S, ip = grp % period; uint32_t ph = (uint32_t)((grp / period) & 1);
        const uint32_t my_full = pl.bar_full + 8u * (uint32_t)(grp * LUT_MAX_STAGES);
        int i_next = grp;                             // local index of this group's next unit
        int i_base = 0;                               // local index of the first unit of the current slab
        for (int64_t slab = slab_beg; slab <= slab_end; ++slab) {
            const int cb0 = (slab == slab_beg) ? (int)(u_beg - slab * n_cblocks) : 0;
            const int cb1 = (slab == slab_end) ? (int)(u_end - slab * n_cblocks) : ncb;
            consumer_bar<CW * 32>();      // everyone finished looking up the previous slab's tables
            if (H2 && TERN) lut_build_h2_tern(pl.tab, v, v1, vbar, vbar1, sc0, sc1, n, slab, tid);
            else if (H2) lut_build_h2(pl.tab, v, v1, vbar, vbar1, sc0, sc1, n, slab, tid);
            else if (TERN) lut_build_tern<CW * 32>(pl.tab, v, vbar, n, slab, tid);
            else lut_build<CW * 32>(pl.tab, v, vbar, n, slab, tid);
            consumer_bar<CW * 32>();
            float* __restrict__ outp = part + ((int64_t)(H2 ? vidx / CPW : 0) * n_slabs + slab) * p_out + col;
            const int i_end = i_base + (cb1 - cb0);
            for (; i_next < i_end; i_next += G) {
                const int cb = cb0 + (i_next - i_base);
                mbar_wait(my_full + 8u * st, ph);
                float sum;
                if constexpr (COL) {
                    const uint32_t a0 = pl.stage(st) + col_off;
                    uint32_t wd[32];
#pragma unroll
                    for (int s = 0; s < 32; ++s) wd[s] = lds_u32(a0 ^ (16u * s + 4u * (s & 3)));
                    // the stage's bytes are now in registers: hand the slot back to the producer
                    __syncwarp();
                    if (lane == 0) mbar_arrive(pl.bar_empty + 8u * st);
                    float ws[32];
#pragma unroll
                    for (int s = 0; s < 32; ++s) {
                        const uint32_t y = y0 ^ (uint32_t)(4 * s * 0x0101);
                        const float t0 = lds_f32(prmt<0xE604u>(wd[s], y));
                        const float t1 = lds_f32(prmt<0xE615u>(wd[s], y));
                        const float t2 = lds_f32(prmt<0xF724u>(wd[s], y));
                        const float t3 = lds_f32(prmt<0xF735u>(wd[s], y));
                        ws[s] = (t0 + t1) + (t2 + t3);
                    }
                    // pairwise tree over the word positions, pairing w with w ^ 8, then ^ 4, ^ 2, ^ 1, ^ 16: the butterfly's
                    // tree (w = w0 ^ s maps it onto itself), so the column sums are bit-identical to the shuffle kernel's
                    // and do not depend on where a column sits in the stage
#pragma unroll
                    for (int k = 0, done = 0; k < 5; ++k) {
                        const int b = (k < 4) ? (8 >> k) : 16;
#pragma unroll
                        for (int s = 0; s < 32; ++s)
                            if ((s & (done | b)) == 0) ws[s] = ws[s] + ws[s | b];
                        done |= b;
                    }
                    sum = ws[0];
                } else {
                    const uint32_t colbase = pl.stage(st) + lane_off;
                    float acc[NACC];
                    uint4 q4 = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
                    for (int c = 0; c < CPW; ++c) {
                        uint32_t w;
                        if (QUAD) {
                            if ((c & 3) == 0) q4 = lds_u128(colbase + ((512u * (c >> 2)) ^ lqs));
                            w = (c & 3) == 0 ? q4.x : (c & 3) == 1 ? q4.y : (c & 3) == 2 ? q4.z : q4.w;
                        } else {
                            w = lds_u32(colbase + 128u * c);
                        }
                        if (!H2) {
                            const float t0 = lds_f32(__byte_perm(w, lb[0], 0x7604));
                            const float t1 = lds_f32(__byte_perm(w, lb[1], 0x7614));
                            const float t2 = lds_f32(__byte_perm(w, lb[2], 0x7624));
                            const float t3 = lds_f32(__byte_perm(w, lb[3], 0x7634));
                            acc[c] = (t0 + t1) + (t2 + t3);
                        } else {
                            const uint32_t r0 = lds_u32(__byte_perm(w, lb[0], 0x7604));
                            const uint32_t r1 = lds_u32(__byte_perm(w, lb[1], 0x7614));
                            const uint32_t r2 = lds_u32(__byte_perm(w, lb[2], 0x7624));
                            const uint32_t r3 = lds_u32(__byte_perm(w, lb[3], 0x7634));
                            const __half2 h = __hadd2(__hadd2(*reinterpret_cast<const __half2*>(&r0), *reinterpret_cast<const __half2*>(&r1)),
                                                      __hadd2(*reinterpret_cast<const __half2*>(&r2), *reinterpret_cast<const __half2*>(&r3)));
                            const float2 f = __half22float2(h);
                            acc[c] = f.x;
                            acc[(H2 ? CPW : 0) + c] = f.y;
                        }
                    }
                    // the stage's bytes are now in registers: hand the slot back to the producer
                    __syncwarp();
                    if (lane == 0) mbar_arrive(pl.bar_empty + 8u * st);
                    if (TERN) {
                        // select-free butterfly (slots pre-arranged, see above): levels NACC/2 .. 1 (NACC = 32 here)
                        int o = NACC / 2;
#pragma unroll
                        for (int h = NACC / 2; h >= 1; h >>= 1, o >>= 1) {
#pragma unroll
                            for (int c = 0; c < h; ++c) acc[c] = acc[c] + __shfl_xor_sync(0xffffffffu, acc[c + h], o);
                        }
                    } else {
                        // butterfly: NACC sums per lane -> one per lane; the high lane bits select the value
                        int o = 16;
#pragma unroll
                        for (int h = NACC / 2; h >= 1; h >>= 1, o >>= 1) {
                            const bool upper = (lane & o) != 0;
#pragma unroll
                            for (int c = 0; c < h; ++c) {
                                const float send = upper ? acc[c] : acc[c + h];
                                const float keep = upper ? acc[c + h] : acc[c];
                                acc[c] = keep + __shfl_xor_sync(0xffffffffu, send, o);
                            }
                        }
#pragma unroll
                        for (int oo = 16 / NACC; oo >= 1; oo >>= 1) acc[0] += __shfl_xor_sync(0xffffffffu, acc[0], oo);
                    }
                    sum = acc[0];
                }
                const int jj = cb * LUT_STAGE_COLS + col;
                if (writer && jj < (int)p_out) outp[cb * LUT_STAGE_COLS] = sum;
                st += G; while (st >= S) st -= S;
                ip += G; if (ip >= period) { ip -= period; ph ^= 1u; }
            }
            i_base = i_end;
        }
    }
}

// the FAST / PAIR sweeps stream the ternary copy when the handle has one (the TMEM variant reads the 2-bit tiles)
bool sweep_tmem_enabled(const ihtb_geno* g);
bool sweep_uses_tern(const ihtb_geno* g) { return g->tern.p != nullptr && g->quad && !sweep_tmem_enabled(g); }
int64_t sweep_fast_num_slabs(const ihtb_geno* g) { return sweep_uses_tern(g) ? g->tern_slabs : g->stride / 128; }

// sweep_tmem.cu: the same sweeps with the genotype stream staged through tensor memory (quad layout only)
bool sweep_tmem_enabled(const ihtb_geno* g);
void sweep_tmem_partials(const ihtb_geno* g, const double* d_v, const double* d_vbar, float* d_part, cudaStream_t s);
void sweep_tmem_pair_partials(const ihtb_geno* g, const double* d_v0, const double* d_v1, const double* d_vbar,
                              const float* d_scale, float* d_part, cudaStream_t s);

template <bool QUAD, bool H2, bool TERN = false>
static void launch_lut(const ihtb_geno* g, const double* d_v, const double* d_v1, const double* d_vbar,
                       const float* d_scale, float* d_part, cudaStream_t s) {
    constexpr int G = (TERN && !H2) ? 4 : 2;         // one column per lane: 4 warps cover a 128-column unit
    ensure_dynamic_smem(k_sweep_lut<16, G, QUAD, H2, TERN>, LUT_SMEM_BYTES);
    const int64_t n_slabs = TERN ? g->tern_slabs : g->stride / 128;
    const int64_t n_cblocks = ceil_div(g->p4, LUT_STAGE_COLS);
    int64_t units = n_slabs * n_cblocks;
    int grid = g->sm_count;
    if (units < grid) grid = (int)units;
    IHTB_CHECK(g->p < (int64_t(1) << 31) - 256, IHTB_EDIM, "more than 2^31 SNP columns on one GPU");
    IHTB_LAUNCH((k_sweep_lut<16, G, QUAD, H2, TERN>), grid, 17 * 32, LUT_SMEM_BYTES, s, TERN ? g->tern.p : g->bed.p, g->cs_j,
                g->cs_s, g->p4, g->p, g->n, n_slabs, d_v, d_v1, d_vbar, d_scale, d_part, (uint32_t)LUT_SMEM_BYTES);
}

// FAST sweep, one right-hand side: d_part is [n_slabs][p] floats
void sweep_fast_partials(const ihtb_geno* g, const double* d_v, const double* d_vbar, float* d_part, int64_t* n_slabs_out,
                         cudaStream_t s) {
    if (n_slabs_out) *n_slabs_out = sweep_fast_num_slabs(g);
    if (sweep_tmem_enabled(g)) { sweep_tmem_partials(g, d_v, d_vbar, d_part, s); return; }
    if (sweep_uses_tern(g)) launch_lut<true, false, true>(g, d_v, nullptr, d_vbar, nullptr, d_part, s);
    else if (g->quad) launch_lut<true, false>(g, d_v, nullptr, d_vbar, nullptr, d_part, s);
    else launch_lut<false, false>(g, d_v, nullptr, d_vbar, nullptr, d_part, s);
}

void sweep_fast_kernel_only(const ihtb_geno* g, const double* d_v, const double* d_vbar, float* d_part, cudaStream_t s) {
    sweep_fast_partials(g, d_v, d_vbar, d_part, nullptr, s);
}

// PAIR sweep, two right-hand sides per pass: d_vbar[2] means, d_scale[2] power-of-two scales (device);
// d_part is [2][n_slabs][p] floats of the scaled sums
void sweep_pair_partials(const ihtb_geno* g, const double* d_v0, const double* d_v1, const double* d_vbar,
                         const float* d_scale, float* d_part, cudaStream_t s) {
    IHTB_CHECK(g->cs_j == 128, IHTB_EUNSUPPORTED, "the pair sweep needs a tiled layout");
    if (sweep_tmem_enabled(g)) { sweep_tmem_pair_partials(g, d_v0, d_v1, d_vbar, d_scale, d_part, s); return; }
    if (sweep_uses_tern(g)) launch_lut<true, true, true>(g, d_v0, d_v1, d_vbar, d_scale, d_part, s);
    else if (g->quad) launch_lut<true, true>(g, d_v0, d_v1, d_vbar, d_scale, d_part, s);
    else launch_lut<false, true>(g, d_v0, d_v1, d_vbar, d_scale, d_part, s);
}

}  // namespace ihtb
