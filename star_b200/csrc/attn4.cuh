// star_b200 / csrc / attn4.cuh
// Spatial-attention kernel (head_dim 64): two 128-row query tiles per CTA share every K/V tile (5-stage TMA ring),
// S = Q K^T in TMEM, single-pass online softmax with lazy rescale, O accumulated in TMEM, and the probabilities kept in
// TENSOR MEMORY:
//   * P_t(j) is written with tcgen05.st as packed fp16 pairs (64 columns per tile) and the PV MMA takes its A operand
//     from TMEM (tcgen05.mma [d], [a_tmem], b_desc).  The ncu capture of the SS formulation (profiles/r01_ncu_attn2.txt)
//     showed the shared-memory port as its limiter (256 KB per KV tile = 2048 clk at 128 B/clk, twice the MMA time);
//     keeping P out of smem halves that.
//   * two MMA-issuing threads (warp 1: query tile 0, warp 2: query tile 1): one independent S -> P -> PV pipeline per
//     tile, descriptors built once and advanced by 64-bit adds.
//   * softmax arithmetic in packed fp32x2 (FFMA2 / FADD2), compile-time specialisation of the ragged last KV tile.
//   * two softmax threads per query row (640 threads): score columns [0,64) / [64,128) of the KV tile, O columns
//     [0,32) / [32,64); the halves agree on the row maximum through shared memory and one 256-thread named barrier
//     per KV tile.  16 softmax warps keep the 16-lane MUFU ~80 % busy (every exponential on the MUFU: the FMA-pipe
//     polynomial share, the two query tiles taking turns on the MUFU and the one-thread-per-row organisation were
//     measured and lost, DESIGN.md section 3).
// TMEM columns: S[t] t*128, O[t] 256 + t*64, P[t] 384 + t*64.
#pragma once
#include "common.cuh"
#include "attn.cuh"

// Instrumented build (tools/build_variant.py -DSTAR_ATTN_TRACE=1; never set in the shipped library):
//   STAR_ATTN_TRACE 1: CTA (0,0,0) records clock64() of the softmax phases of both tiles per KV step (tools/attn_trace.py).
#ifndef STAR_ATTN_TRACE
#define STAR_ATTN_TRACE 0
#endif

namespace star {

STAR_DEVINL void a4_st_shared_f32(uint32_t addr, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory"); }
STAR_DEVINL float a4_ld_shared_f32(uint32_t addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
    return v;
}
STAR_DEVINL void a4_named_bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

#if STAR_ATTN_TRACE
__device__ long long g_a4_trace[2][8192];          // [query tile][slot]: (event, clock) pairs of warp 4 / warp 12 lane 0
__device__ int g_a4_trace_n[2];
STAR_DEVINL void a4_trace(int t, int event, int& i) {      // the slot counter lives in a register: an event costs ~2 stores
    if (i + 1 < 8192) {
        long long c;
        asm volatile("mov.u64 %0, %%clock64;" : "=l"(c)::"memory");
        g_a4_trace[t][i] = event;
        g_a4_trace[t][i + 1] = c;
        i += 2;
        g_a4_trace_n[t] = i;
    }
}
#define A4_TRACE(ev) do { if (trace_me) a4_trace(t, ev, trace_i); } while (0)
#else
#define A4_TRACE(ev)
#endif

struct TagFalse { static constexpr bool value = false; };
struct TagTrue { static constexpr bool value = true; };

constexpr int A4S_THREADS = 640;     // warps 0-3: TMA, MMA x2, idle; warps 4-11 query tile 0 (4-7 low score half, 8-11 high half), 12-19 query tile 1
constexpr int A4_KV_STAGES = 5;

struct Attn4Smem {
    static constexpr int TILE = 128 * 64 * 2;                 // 16 KB
    static constexpr int OFF_Q = 0;                           // 2 tiles
    static constexpr int OFF_K = OFF_Q + 2 * TILE;
    static constexpr int OFF_V = OFF_K + A4_KV_STAGES * TILE;
    static constexpr int OFF_X = OFF_V + A4_KV_STAGES * TILE; // SPLIT exchange: float [2 tiles][2 parity][2 halves][128]
    static constexpr int OFF_BAR = OFF_X + 2 * 2 * 2 * 128 * 4;
    static constexpr int TOTAL = OFF_BAR + 256 + 1024;
};

__global__ void __launch_bounds__(A4S_THREADS, 1)
attn4_fwd_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_k,
                 const __grid_constant__ CUtensorMap tmap_v, const __grid_constant__ AttnParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Attn4Smem::OFF_BAR);
    uint64_t* q_full = bars;                 // 1
    uint64_t* kv_full = bars + 1;            // 5
    uint64_t* kv_empty = bars + 6;           // 5
    uint64_t* s_full = bars + 11;            // 2   MMA -> softmax WG t : S_t(j) complete
    uint64_t* s_free = bars + 13;            // 2   softmax WG t -> MMA : S_t(j) is in registers
    uint64_t* p_full = bars + 15;            // 2   softmax WG t -> MMA : P_t(j) in TMEM, O_t rescaled
    uint64_t* pv_done = bars + 17;           // 2   MMA -> softmax WG t : O_t += P_t(j) V_j retired
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 19);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int q0 = blockIdx.x * 256;
    const int head = blockIdx.y;
    const int batch = blockIdx.z;
    const int kv_batch = batch / p.kv_batch_div;
    const int nt = (p.Nk + 127) / 128;
    const int ntq = (q0 + 128 < p.Nq) ? 2 : 1;          // second query tile may be empty

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmap_q);
        tma_prefetch_desc(&tmap_k);
        tma_prefetch_desc(&tmap_v);
    }
    if (warp == 1) {
        if (lane == 0) {
            mbar_init(q_full, 1);
            for (int s = 0; s < A4_KV_STAGES; ++s) {
                mbar_init(&kv_full[s], 1);
                mbar_init(&kv_empty[s], ntq > 1 ? 2 : 1);
            }
            for (int t = 0; t < 2; ++t) {
                mbar_init(&s_full[t], 1);
                mbar_init(&s_free[t], 256);
                mbar_init(&p_full[t], 256);
                mbar_init(&pv_done[t], 1);
            }
            fence_barrier_init();
        }
        __syncwarp();
        tmem_alloc<512>(tmem_slot);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;      // S[t] at cols t*128, O[t] at cols 256 + t*64

    if (warp == 0) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
        if (lane == 0) {
            mbar_expect_tx(q_full, ntq * Attn4Smem::TILE);
            for (int t = 0; t < ntq; ++t)
                tma_load_3d(smem + Attn4Smem::OFF_Q + t * Attn4Smem::TILE, &tmap_q, q_full, head * 64, q0 + t * 128, batch);
            for (int j = 0; j < nt; ++j) {
                const int s = j % A4_KV_STAGES;
                mbar_wait(&kv_empty[s], ((j / A4_KV_STAGES) & 1) ^ 1);
                mbar_expect_tx(&kv_full[s], 2 * Attn4Smem::TILE);
                tma_load_3d(smem + Attn4Smem::OFF_K + s * Attn4Smem::TILE, &tmap_k, &kv_full[s], head * 64, j * 128, kv_batch);
                tma_load_3d(smem + Attn4Smem::OFF_V + s * Attn4Smem::TILE, &tmap_v, &kv_full[s], head * 64, j * 128, kv_batch);
            }
        }
    } else if (warp == 1) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
        if (lane == 0) {
            constexpr uint32_t idesc_s = umma_idesc_f16(128, 128, 0, 0);
            constexpr uint32_t idesc_o = umma_idesc_f16(128, 64, 0, 1);
            // descriptors are built once; a stage / k-step is a 64-bit add (the issuing threads are on the critical path)
            const uint64_t dq0 = umma_desc_sw128(smem_u32(smem + Attn4Smem::OFF_Q), 16, 1024);
            const uint64_t dk0 = umma_desc_sw128(smem_u32(smem + Attn4Smem::OFF_K), 16, 1024);
            const uint64_t dv0 = umma_desc_sw128(smem_u32(smem + Attn4Smem::OFF_V), 8192, 1024);
            constexpr uint64_t TILE_INC = (uint64_t)(Attn4Smem::TILE >> 4);
            auto issue_s = [&](int t, int j) {
                const uint64_t dq = dq0 + TILE_INC * (uint64_t)t;
                const uint64_t dk = dk0 + TILE_INC * (uint64_t)(j % A4_KV_STAGES);
                umma_f16_ss(tmem_base + t * 128, dq, dk, idesc_s, 0u);
                umma_f16_ss(tmem_base + t * 128, dq + 2, dk + 2, idesc_s, 1u);
                umma_f16_ss(tmem_base + t * 128, dq + 4, dk + 4, idesc_s, 1u);
                umma_f16_ss(tmem_base + t * 128, dq + 6, dk + 6, idesc_s, 1u);
                umma_commit(&s_full[t]);
            };
            mbar_wait(q_full, 0);
            mbar_wait(&kv_full[0], 0);
            tc_fence_after();
            issue_s(0, 0);
            auto issue_pv = [&](int t, int j) {
                mbar_wait(&p_full[t], j & 1);
                tc_fence_after();
                const uint64_t dv = dv0 + TILE_INC * (uint64_t)(j % A4_KV_STAGES);
                const uint32_t d_o = tmem_base + 256 + t * 64, a_p = tmem_base + 384 + t * 64;
#pragma unroll
                for (int k = 0; k < 8; ++k)             // A = P_t (TMEM, 8 columns = 16 fp16 keys per step), B = V (MN-major)
                    umma_f16_ts(d_o, a_p + k * 8, dv + (uint64_t)(k * 128), idesc_o, (j > 0 || k > 0) ? 1u : 0u);
                umma_commit(&pv_done[t]);
            };
            auto next_s = [&](int t, int j) {           // S_t(j+1) as soon as S_t(j) sits in the softmax registers
                mbar_wait(&s_free[t], j & 1);
                tc_fence_after();
                issue_s(t, j + 1);
            };
            // independent pipeline per query tile: this thread only drives tile 0 (warp 2 drives tile 1)
            for (int j = 0; j < nt; ++j) {
                if (j + 1 < nt) {
                    mbar_wait(&kv_full[(j + 1) % A4_KV_STAGES], ((j + 1) / A4_KV_STAGES) & 1);
                    next_s(0, j);
                }
                issue_pv(0, j);
                umma_commit(&kv_empty[j % A4_KV_STAGES]);
            }
        }
    } else if (warp < 4) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
        if (warp == 2 && lane == 0 && ntq > 1) {
            // second MMA-issuing thread: query tile 1
            constexpr uint32_t idesc_s = umma_idesc_f16(128, 128, 0, 0);
            constexpr uint32_t idesc_o = umma_idesc_f16(128, 64, 0, 1);
            const uint64_t dq = umma_desc_sw128(smem_u32(smem + Attn4Smem::OFF_Q + Attn4Smem::TILE), 16, 1024);
            const uint64_t dk0 = umma_desc_sw128(smem_u32(smem + Attn4Smem::OFF_K), 16, 1024);
            const uint64_t dv0 = umma_desc_sw128(smem_u32(smem + Attn4Smem::OFF_V), 8192, 1024);
            constexpr uint64_t TILE_INC = (uint64_t)(Attn4Smem::TILE >> 4);
            auto issue_s1 = [&](int j) {
                const uint64_t dk = dk0 + TILE_INC * (uint64_t)(j % A4_KV_STAGES);
                umma_f16_ss(tmem_base + 128, dq, dk, idesc_s, 0u);
                umma_f16_ss(tmem_base + 128, dq + 2, dk + 2, idesc_s, 1u);
                umma_f16_ss(tmem_base + 128, dq + 4, dk + 4, idesc_s, 1u);
                umma_f16_ss(tmem_base + 128, dq + 6, dk + 6, idesc_s, 1u);
                umma_commit(&s_full[1]);
            };
            mbar_wait(q_full, 0);
            mbar_wait(&kv_full[0], 0);
            tc_fence_after();
            issue_s1(0);
            for (int j = 0; j < nt; ++j) {
                if (j + 1 < nt) {
                    mbar_wait(&kv_full[(j + 1) % A4_KV_STAGES], ((j + 1) / A4_KV_STAGES) & 1);
                    mbar_wait(&s_free[1], j & 1);
                    tc_fence_after();
                    issue_s1(j + 1);
                }
                mbar_wait(&p_full[1], j & 1);
                tc_fence_after();
                const uint64_t dv = dv0 + TILE_INC * (uint64_t)(j % A4_KV_STAGES);
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    umma_f16_ts(tmem_base + 256 + 64, tmem_base + 384 + 64 + k * 8, dv + (uint64_t)(k * 128), idesc_o,
                                (j > 0 || k > 0) ? 1u : 0u);
                umma_commit(&pv_done[1]);
                umma_commit(&kv_empty[j % A4_KV_STAGES]);
            }
        }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 104;");
        const int t = (warp - 4) >> 3;                   // query tile
        const int half = ((warp - 4) >> 2) & 1;          // score columns [64*half, +64) of every KV tile, O columns [32*half, +32)
        if (t < ntq) {
            const int quad = warp & 3;
            const int r = quad * 32 + lane;
            const uint32_t lane_off = (uint32_t)(quad * 32) << 16;
            const uint32_t t_s = tmem_base + t * 128 + half * 64 + lane_off;
            const uint32_t t_o = tmem_base + 256 + t * 64 + half * 32 + lane_off;
            const uint32_t t_p = tmem_base + 384 + t * 64 + half * 32 + lane_off;     // 64 probabilities = 32 packed columns
            const uint32_t x_base = smem_u32(smem + Attn4Smem::OFF_X) + (uint32_t)t * 2048u;    // [parity][half][row]
            const int bar_id = 1 + t;
            const float sl2 = p.scale_log2;
            float m_used = 0.f, l_run = 0.f;
#if STAR_ATTN_TRACE
            const bool trace_me = blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && half == 0 && quad == 0 && lane == 0;
            int trace_i = 0;
#endif
            auto kv_tile = [&](const int j, auto tail_tag) {
                constexpr bool tail = decltype(tail_tag)::value;
                const int kbase = j * 128 + half * 64;
                A4_TRACE(1);
                mbar_wait(&s_full[t], j & 1);
                tc_fence_after();
                A4_TRACE(2);
                uint32_t v[64];
                tmem_ld32(t_s, v);
                tmem_ld32(t_s + 32, v + 32);
                tmem_ld_wait();
                tc_fence_before();
                mbar_arrive(&s_free[t]);
                A4_TRACE(3);
                if (tail) {
#pragma unroll
                    for (int i = 0; i < 64; ++i)
                        if (kbase + i >= p.Nk) v[i] = 0xff800000u;      // -inf
                }
                float m0 = -INFINITY, m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;
#pragma unroll
                for (int i = 0; i < 64; i += 8) {
                    m0 = fmaxf(m0, fmaxf(__uint_as_float(v[i]), __uint_as_float(v[i + 1])));
                    m1 = fmaxf(m1, fmaxf(__uint_as_float(v[i + 2]), __uint_as_float(v[i + 3])));
                    m2 = fmaxf(m2, fmaxf(__uint_as_float(v[i + 4]), __uint_as_float(v[i + 5])));
                    m3 = fmaxf(m3, fmaxf(__uint_as_float(v[i + 6]), __uint_as_float(v[i + 7])));
                }
                const float mx_mine = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
                const uint32_t x_slot = x_base + (uint32_t)(j & 1) * 1024u;
                a4_st_shared_f32(x_slot + (uint32_t)half * 512u + (uint32_t)r * 4u, mx_mine);
                a4_named_bar_sync(bar_id, 256);
                const float mx = fmaxf(mx_mine, a4_ld_shared_f32(x_slot + (uint32_t)(half ^ 1) * 512u + (uint32_t)r * 4u));
                A4_TRACE(4);
                const float mc = mx * sl2;
                float factor = 1.f;
                bool need = false;
                if (j == 0) {
                    m_used = mc;
                } else if (mc > m_used + 8.0f) {
                    factor = ex2_approx(m_used - mc);
                    m_used = mc;
                    need = true;
                }
                uint64_t l0 = 0ull, l1 = 0ull;
                uint32_t pk[32];
                const uint64_t sl2_2 = f2_pack(sl2, sl2), negm_2 = f2_pack(-m_used, -m_used);
#pragma unroll
                for (int e = 0; e < 32; ++e) {
                    const int i = e * 2;
                    const uint64_t x01 = f2_fma(f2_pack_bits(v[i], v[i + 1]), sl2_2, negm_2);
                    float x0, x1;
                    f2_unpack(x01, x0, x1);
                    const uint64_t p01 = f2_pack(ex2_approx(x0), ex2_approx(x1));
                    float p0, p1;
                    f2_unpack(p01, p0, p1);
                    pk[e] = pack_half2(p0, p1);
                    if (e & 1) l1 = f2_add(l1, p01);
                    else l0 = f2_add(l0, p01);
                }
                float l_lo, l_hi;
                f2_unpack(f2_add(l0, l1), l_lo, l_hi);
                A4_TRACE(5);
                if (j > 0) {
                    mbar_wait(&pv_done[t], (j - 1) & 1);         // P buffer free, O_t stable
                    tc_fence_after();
                    A4_TRACE(6);
                    if (__any_sync(0xffffffffu, need)) {
                        uint32_t o[32];
                        tmem_ld32(t_o, o);
                        tmem_ld_wait();
#pragma unroll
                        for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * factor);
                        tmem_st32(t_o, o);
                        tmem_st_wait();
                        l_run *= factor;
                    }
                }
                tmem_st32(t_p, pk);
                tmem_st_wait();
                tc_fence_before();
                mbar_arrive(&p_full[t]);
                A4_TRACE(7);
                l_run += l_lo + l_hi;
            };
#pragma unroll 1
            for (int j = 0; j < nt - 1; ++j) kv_tile(j, TagFalse{});
            if (p.Nk & 127) kv_tile(nt - 1, TagTrue{});
            else kv_tile(nt - 1, TagFalse{});
            // combine the two halves' row sums, then O / l -> fp16 (each thread stores its 32 output columns)
            const uint32_t x_slot = x_base + (uint32_t)(nt & 1) * 1024u;
            a4_st_shared_f32(x_slot + (uint32_t)half * 512u + (uint32_t)r * 4u, l_run);
            a4_named_bar_sync(bar_id, 256);
            const float l_tot = l_run + a4_ld_shared_f32(x_slot + (uint32_t)(half ^ 1) * 512u + (uint32_t)r * 4u);
            mbar_wait(&pv_done[t], (nt - 1) & 1);
            tc_fence_after();
            const int q = q0 + t * 128 + r;
            const float inv = 1.0f / l_tot;
            uint32_t o[32];
            tmem_ld32(t_o, o);
            tmem_ld_wait();
            if (q < p.Nq) {
                __half* op = p.out + ((long long)batch * p.Nq + q) * p.ldo + head * 64 + half * 32;
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    uint4 w;
                    w.x = pack_half2(__uint_as_float(o[u * 8 + 0]) * inv, __uint_as_float(o[u * 8 + 1]) * inv);
                    w.y = pack_half2(__uint_as_float(o[u * 8 + 2]) * inv, __uint_as_float(o[u * 8 + 3]) * inv);
                    w.z = pack_half2(__uint_as_float(o[u * 8 + 4]) * inv, __uint_as_float(o[u * 8 + 5]) * inv);
                    w.w = pack_half2(__uint_as_float(o[u * 8 + 6]) * inv, __uint_as_float(o[u * 8 + 7]) * inv);
                    reinterpret_cast<uint4*>(op)[u] = w;
                }
            }
            tc_fence_before();
        }
    }
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc<512>(tmem_base);
    }
}

}  // namespace star
