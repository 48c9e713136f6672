// star_b200 / csrc / common.cuh
// sm_100a device helpers: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc /
// mma / commit / ld), UMMA shared-memory + instruction descriptors.  Raw PTX;
// bit layouts follow the PTX ISA "tcgen05 matrix descriptors" tables (cross-checked
// against cute/arch/mma_sm100_desc.hpp field positions).
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

// One source, two builds: libstar_sm100.so computes on fp16 tokens, libstar_sm100_bf16.so (-DSTAR_BF16) on bf16 tokens
// (the CogVideoX DiT runs bf16: cogvideox_5b_infer_sr.yaml:11).  Every storage-type conversion in the kernels goes through
// the intrinsics re-pointed below; accumulation, statistics and softmax stay fp32 in both builds.
#ifdef STAR_BF16
#include <cuda_bf16.h>
#define __half __nv_bfloat16
#define __half2 __nv_bfloat162
#define __float2half_rn __float2bfloat16_rn
#define __half2float __bfloat162float
#define __floats2half2_rn __floats2bfloat162_rn
#define __half22float2 __bfloat1622float2
#define STAR_UMMA_FMT 1u                                   /* tcgen05 kind::f16 A/B format: 1 = bf16 */
#define STAR_TMAP_DTYPE CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
#define STAR_MMA_SYNC_T "bf16"
#else
#define STAR_UMMA_FMT 0u                                   /* 0 = fp16 */
#define STAR_TMAP_DTYPE CU_TENSOR_MAP_DATA_TYPE_FLOAT16
#define STAR_MMA_SYNC_T "f16"
#endif

namespace star {

#define STAR_DEVINL __device__ __forceinline__

STAR_DEVINL uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---------------------------------------------------------------- mbarrier
STAR_DEVINL void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
STAR_DEVINL void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
STAR_DEVINL void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
STAR_DEVINL void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
STAR_DEVINL bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred P;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, P;\n\t}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug (lost arrive / wrong parity) traps after ~2 s of SM clocks instead of hanging
// the GPU (try_wait itself may block for a system-dependent time, so the bound is on clock64, not on spins).
#ifndef STAR_WAIT_CYCLES
#define STAR_WAIT_CYCLES 4000000000ll
#endif
STAR_DEVINL void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    long long t0 = 0;
    while (!mbar_try_wait(bar, parity)) {
        if ((++spins & 255u) == 0) {
            const long long now = clock64();
            if (t0 == 0) {
                t0 = now;
            } else if (now - t0 > STAR_WAIT_CYCLES) {
                printf("star: mbarrier wait timed out (block %d,%d,%d thread %d bar smem+0x%x parity %u)\n", blockIdx.x,
                       blockIdx.y, blockIdx.z, threadIdx.x, smem_u32(bar), parity);
                __trap();
            }
        }
    }
}

// ---------------------------------------------------------------- fences
STAR_DEVINL void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
STAR_DEVINL void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
STAR_DEVINL void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---------------------------------------------------------------- TMA
STAR_DEVINL void tma_prefetch_desc(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
STAR_DEVINL void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
STAR_DEVINL void tma_load_3d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
STAR_DEVINL void tma_load_5d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3, int c4) {
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2),
        "r"(c3), "r"(c4)
        : "memory");
}

// ---------------------------------------------------------------- TMEM
template <uint32_t kCols>
STAR_DEVINL void tmem_alloc(uint32_t* dst_in_smem) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_in_smem)),
                 "n"(kCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
STAR_DEVINL void tmem_dealloc(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}

// 32 lanes x 32 consecutive 32-bit columns -> 32 registers per thread (thread i = lane i of the warp's quadrant)
STAR_DEVINL void tmem_ld32(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
STAR_DEVINL void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------- UMMA descriptors
// Shared-memory matrix descriptor (64-bit):
//   [0,14)  start address >> 4          [16,30) leading-dim byte offset >> 4
//   [32,46) stride-dim byte offset >> 4 [46,48) version = 1 (sm_100)
//   [49,52) base offset = 0             [61,64) layout: 0 none, 2 = SWIZZLE_128B
// K-major, SWIZZLE_128B canonical tile = rows of 128 B, 8-row groups of 1024 B
// (exactly what TMA SWIZZLE_128B writes for a box with a 128-byte inner extent):
//   SBO = 1024 B (distance between 8-row groups), LBO unused for swizzled K-major.
// MN-major, SWIZZLE_128B ([k][mn] with 64 mn-elements = 128 B contiguous per k row):
//   8 k-rows form a 1024 B atom; SBO = 1024 B between k-groups of 8; LBO = distance
//   between 64-element mn blocks.
STAR_DEVINL uint64_t umma_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

// Instruction descriptor for kind::f16 (fp16 A/B, fp32 accumulate):
//   [4,6) D fmt: 1 = f32   [7,10) A fmt: 0 = f16, 1 = bf16   [10,13) B fmt: same
//   [15] A major (0 = K)   [16] B major (0 = K, 1 = MN)
//   [17,23) N >> 3         [24,29) M >> 4
STAR_DEVINL constexpr uint32_t umma_idesc_f16(uint32_t M, uint32_t N, uint32_t a_mn_major, uint32_t b_mn_major) {
    return (1u << 4) | (STAR_UMMA_FMT << 7) | (STAR_UMMA_FMT << 10) | (a_mn_major << 15) | (b_mn_major << 16) | ((N >> 3) << 17) |
           ((M >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread.
STAR_DEVINL void umma_f16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}

// D[tmem] (+)= A[tmem] * B[smem]: A = 128 lanes x (K/2) 32-bit columns of packed 16-bit pairs
STAR_DEVINL void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n"
        ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}

// mbarrier arrives once all previously issued tcgen05.mma of this thread have completed
// (implies tcgen05.fence::before_thread_sync).
STAR_DEVINL void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}

// ---------------------------------------------------------------- misc math
STAR_DEVINL float ex2_approx(float x);
STAR_DEVINL float silu_f(float x) { return x / (1.0f + __expf(-x)); }
// exact (erf) GELU, nn.GELU() default (unet_v2v.py:504).  erf by Abramowitz-Stegun 7.1.26 (|err| <= 1.5e-7, far
// below the fp16 rounding of the result): 2 MUFU + ~12 FMA-pipe ops instead of libdevice erff's ~30.
STAR_DEVINL float erf_as(float x) {
    const float ax = fabsf(x);
    float t;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, ax, 1.0f)));
    float poly = fmaf(1.061405429f, t, -1.453152027f);
    poly = fmaf(poly, t, 1.421413741f);
    poly = fmaf(poly, t, -0.284496736f);
    poly = fmaf(poly, t, 0.254829592f);
    const float e = ex2_approx(-1.4426950408889634f * ax * ax);
    const float r = fmaf(-poly * t, e, 1.0f);
    return copysignf(r, x);
}
STAR_DEVINL float gelu_erf_f(float x) { return 0.5f * x * (1.0f + erf_as(x * 0.70710678118654752f)); }
STAR_DEVINL float gelu_tanh_f(float x) {
    const float u = 0.7978845608028654f * (x + 0.044715f * x * x * x);
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(u));
    return 0.5f * x * (1.0f + t);
}
STAR_DEVINL float sigmoid_f(float x) { return 1.0f / (1.0f + __expf(-x)); }

STAR_DEVINL uint32_t pack_half2(float a, float b) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}

}  // namespace star

namespace star {
// 32 lanes x 32 columns: registers -> TMEM (thread i writes lane i of the warp's quadrant)
STAR_DEVINL void tmem_st32(uint32_t taddr, const uint32_t* r) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
        "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
        "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
}
STAR_DEVINL void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

STAR_DEVINL void unpack8h(const uint4& u, float* f) {
    const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 t = __half22float2(h[i]);
        f[2 * i] = t.x;
        f[2 * i + 1] = t.y;
    }
}

STAR_DEVINL float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// ---- packed fp32x2 arithmetic (sm_100: FFMA2 / FADD2, one issue slot for two lanes' worth of work) ----
STAR_DEVINL uint64_t f2_pack(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
STAR_DEVINL uint64_t f2_pack_bits(uint32_t lo, uint32_t hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi));
    return r;
}
STAR_DEVINL void f2_unpack(uint64_t v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
STAR_DEVINL uint64_t f2_fma(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t r;
    asm("fma.rn.ftz.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
STAR_DEVINL uint64_t f2_add(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("add.rn.ftz.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
}  // namespace star
