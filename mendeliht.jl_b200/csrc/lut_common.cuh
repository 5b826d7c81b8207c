// Shared pieces of the table-driven FAST sweeps (sweep_lut.cu: TMA stage ring; sweep_ldg.cu: register-prefetched
// global loads): PTX wrappers and the per-slab table build.
#pragma once
#include "common.cuh"
#include <cuda_fp16.h>

namespace ihtb {

constexpr int LUT_TABLE_BYTES = 131072;

// ---- PTX wrappers ---------------------------------------------------------------------------------
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
__device__ __forceinline__ float lds_f32(uint32_t addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint4 lds_u128(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
// byte permute with the selector as an immediate: unlike __byte_perm, a selector nibble with bit 3 set replicates the
// sign bit of the selected byte (0x00 for a byte below 0x80)
template <uint32_t SEL>
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b) {
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "n"(SEL));
    return d;
}
__device__ __forceinline__ void sts_u32(uint32_t addr, uint32_t v) {
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ void sts_f32(uint32_t addr, float v) {
    asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
template <int NT>
__device__ __forceinline__ void consumer_bar() {   // named barrier 1 over the NT consumer threads
    asm volatile("bar.sync 1, %0;" ::"n"(NT) : "memory");
}

// build T for one slab; executed by the NT (256 or 512) consumer threads
template <int NT>
__device__ __forceinline__ void lut_build(uint32_t tab, const double* __restrict__ v, double vbar, int64_t n,
                                          int64_t slab, int tid) {
    // thread -> (part, group): group = t*32 + w (128 groups); part selects a range of the top sample's code v3
    constexpr int PARTS = NT / 128;          // 2 or 4
    constexpr int V3_PER = 4 / PARTS;        // 2 or 1
    const int group = tid & 127, part = tid >> 7;
    const int t = group >> 5, w = group & 31;
    float u[4];
#pragma unroll
    for (int s = 0; s < 4; ++s) {
        int64_t i = slab * 512 + 16 * w + 4 * t + s;
        u[s] = (i < n) ? __double2float_rn(__dsub_rn(v[i], vbar)) : 0.0f;
    }
    // dosage table of one sample: codes 00, 01 (missing -> 0), 10, 11
    auto f = [&](int s, int code) -> float { return code == 2 ? u[s] : (code == 3 ? u[s] + u[s] : 0.0f); };
    // address of row `value`: window(t>>1) + value*256 + (t&1)*128 + 4*w
    const uint32_t rowbase = tab + (uint32_t)(t >> 1) * 65536u + (uint32_t)(t & 1) * 128u + 4u * (uint32_t)w;
#pragma unroll
    for (int c3 = 0; c3 < V3_PER; ++c3) {
        const int v3 = part * V3_PER + c3;                 // runtime, but only used arithmetically
        const float a3 = (v3 == 2) ? u[3] : ((v3 == 3) ? u[3] + u[3] : 0.0f);
        const uint32_t base3 = rowbase + (uint32_t)v3 * (64u * 256u);
#pragma unroll
        for (int v2 = 0; v2 < 4; ++v2) {
            const float a2 = a3 + f(2, v2);
#pragma unroll
            for (int v1 = 0; v1 < 4; ++v1) {
                const float a1 = a2 + f(1, v1);
#pragma unroll
                for (int v0 = 0; v0 < 4; ++v0)
                    sts_f32(base3 + (uint32_t)(v2 << 4 | v1 << 2 | v0) * 256u, a1 + f(0, v0));
            }
        }
    }
}

// Ternary tiles (ihtb_geno::tern): a byte is five base-3 dosages, a chunk covers 640 samples, word w holds samples
// 20 w .. 20 w + 19 and byte t of it samples 20 w + 5 t .. + 4.  Same table addressing, 243 rows used.  Parts 0..2 take
// one value of the top digit each (81 rows); a fourth part idles.
template <int NT>
__device__ __forceinline__ void lut_build_tern(uint32_t tab, const double* __restrict__ v, double vbar, int64_t n,
                                               int64_t slab, int tid) {
    static_assert(NT == 512, "ternary tables are built by 512 threads");
    const int group = tid & 127, d4 = tid >> 7;
    if (d4 > 2) return;
    const int t = group >> 5, w = group & 31;
    float u[5];
#pragma unroll
    for (int s = 0; s < 5; ++s) {
        int64_t i = slab * 640 + 20 * w + 5 * t + s;
        u[s] = (i < n) ? __double2float_rn(__dsub_rn(v[i], vbar)) : 0.0f;
    }
    auto f = [&](int s, int d) -> float { return d == 1 ? u[s] : (d == 2 ? u[s] + u[s] : 0.0f); };
    const uint32_t rowbase = tab + (uint32_t)(t >> 1) * 65536u + (uint32_t)(t & 1) * 128u + 4u * (uint32_t)w;
    const float a4 = (d4 == 1) ? u[4] : ((d4 == 2) ? u[4] + u[4] : 0.0f);
    const uint32_t base4 = rowbase + (uint32_t)d4 * (81u * 256u);
#pragma unroll
    for (int d3 = 0; d3 < 3; ++d3) {
        const float a3 = a4 + f(3, d3);
#pragma unroll
        for (int d2 = 0; d2 < 3; ++d2) {
            const float a2 = a3 + f(2, d2);
#pragma unroll
            for (int d1 = 0; d1 < 3; ++d1) {
                const float a1 = a2 + f(1, d1);
#pragma unroll
                for (int d0 = 0; d0 < 3; ++d0)
                    sts_f32(base4 + (uint32_t)(27 * d3 + 9 * d2 + 3 * d1 + d0) * 256u, a1 + f(0, d0));
            }
        }
    }
}

__device__ __forceinline__ void lut_build_h2_tern(uint32_t tab, const double* __restrict__ v0, const double* __restrict__ v1,
                                                  double vbar0, double vbar1, float sc0, float sc1, int64_t n, int64_t slab,
                                                  int tid) {
    const int group = tid & 127, d4 = tid >> 7;
    if (d4 > 2) return;
    const int t = group >> 5, w = group & 31;
    float a[5], b[5];
#pragma unroll
    for (int s = 0; s < 5; ++s) {
        int64_t i = slab * 640 + 20 * w + 5 * t + s;
        const float x0 = (i < n) ? __double2float_rn(__dsub_rn(v0[i], vbar0)) * sc0 : 0.0f;     // power-of-two scale: exact
        const float x1 = (i < n) ? __double2float_rn(__dsub_rn(v1[i], vbar1)) * sc1 : 0.0f;
        // word positions 16..31 keep the two right-hand sides in swapped halves: the first butterfly level of the sweep
        // (lane l with l ^ 16) then separates them without a select
        a[s] = (w & 16) ? x1 : x0;
        b[s] = (w & 16) ? x0 : x1;
    }
    auto fa = [&](int s, int d) -> float { return d == 1 ? a[s] : (d == 2 ? a[s] + a[s] : 0.0f); };
    auto fb = [&](int s, int d) -> float { return d == 1 ? b[s] : (d == 2 ? b[s] + b[s] : 0.0f); };
    const uint32_t rowbase = tab + (uint32_t)(t >> 1) * 65536u + (uint32_t)(t & 1) * 128u + 4u * (uint32_t)w;
    const float a4 = fa(4, d4), b4 = fb(4, d4);
    const uint32_t base4 = rowbase + (uint32_t)d4 * (81u * 256u);
#pragma unroll
    for (int d3 = 0; d3 < 3; ++d3) {
        const float a3 = a4 + fa(3, d3), b3 = b4 + fb(3, d3);
#pragma unroll
        for (int d2 = 0; d2 < 3; ++d2) {
            const float a2 = a3 + fa(2, d2), b2 = b3 + fb(2, d2);
#pragma unroll
            for (int d1 = 0; d1 < 3; ++d1) {
                const float a1 = a2 + fa(1, d1), b1 = b2 + fb(1, d1);
#pragma unroll
                for (int d0 = 0; d0 < 3; ++d0) {
                    const __half2 h = __floats2half2_rn(a1 + fa(0, d0), b1 + fb(0, d0));
                    sts_u32(base4 + (uint32_t)(27 * d3 + 9 * d2 + 3 * d1 + d0) * 256u, *reinterpret_cast<const uint32_t*>(&h));
                }
            }
        }
    }
}

// half2 table of one slab for TWO right-hand sides (the pair sweep): entry = (v0 part | v1 part), each the FP32 sum of
// up to four scaled values rounded once to FP16; same addressing as lut_build.  512 consumer threads.
__device__ __forceinline__ void lut_build_h2(uint32_t tab, const double* __restrict__ v0, const double* __restrict__ v1,
                                             double vbar0, double vbar1, float sc0, float sc1, int64_t n, int64_t slab,
                                             int tid) {
    const int group = tid & 127, part = tid >> 7;            // 4 parts: one value of the top sample's code each
    const int t = group >> 5, w = group & 31;
    float a[4], b[4];
#pragma unroll
    for (int s = 0; s < 4; ++s) {
        int64_t i = slab * 512 + 16 * w + 4 * t + s;
        a[s] = (i < n) ? __double2float_rn(__dsub_rn(v0[i], vbar0)) * sc0 : 0.0f;     // power-of-two scale: exact
        b[s] = (i < n) ? __double2float_rn(__dsub_rn(v1[i], vbar1)) * sc1 : 0.0f;
    }
    auto fa = [&](int s, int code) -> float { return code == 2 ? a[s] : (code == 3 ? a[s] + a[s] : 0.0f); };
    auto fb = [&](int s, int code) -> float { return code == 2 ? b[s] : (code == 3 ? b[s] + b[s] : 0.0f); };
    const uint32_t rowbase = tab + (uint32_t)(t >> 1) * 65536u + (uint32_t)(t & 1) * 128u + 4u * (uint32_t)w;
    const int v3 = part;
    const float a3 = fa(3, v3), b3 = fb(3, v3);
    const uint32_t base3 = rowbase + (uint32_t)v3 * (64u * 256u);
#pragma unroll
    for (int v2 = 0; v2 < 4; ++v2) {
        const float a2 = a3 + fa(2, v2), b2 = b3 + fb(2, v2);
#pragma unroll
        for (int v1c = 0; v1c < 4; ++v1c) {
            const float a1 = a2 + fa(1, v1c), b1 = b2 + fb(1, v1c);
#pragma unroll
            for (int v0c = 0; v0c < 4; ++v0c) {
                const __half2 h = __floats2half2_rn(a1 + fa(0, v0c), b1 + fb(0, v0c));
                sts_u32(base3 + (uint32_t)(v2 << 4 | v1c << 2 | v0c) * 256u, *reinterpret_cast<const uint32_t*>(&h));
            }
        }
    }
}

}  // namespace ihtb
