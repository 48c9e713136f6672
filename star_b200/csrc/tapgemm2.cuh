// star_b200 / csrc / tapgemm2.cuh
// Persistent tap-GEMM (same contraction as tapgemm.cuh, see there for the tap / box addressing):
//   * one CTA per SM loops over output tiles (n fastest, so concurrently running CTAs share the A tile in L2)
//   * TMEM holds TWO accumulators: the epilogue of tile i runs while the MMAs of tile i+1 are issued
//   * the epilogue is fully coalesced: residual tile arrives by TMA (prefetched during the main loop),
//     results are staged in swizzled shared memory and leave through TMA stores (hardware clips ragged
//     tile edges and the N tail), bias / time-embedding rows are read with 128-bit loads
// Tile widths BN = 128 / 160 / 256 (star_abi.cu picks: 256 wherever the padded width wastes little; 6 / 5 / 4 operand
// stages).  Warp roles (384 threads): warp 0 TMA producer, warp 1 MMA issuer + TMEM owner, warp 2 idle, warp 3 TMA-STORE thread
// (round 2: the role timeline of one CTA, profiles/r02_gemm_trace_qkv_before.log, showed the epilogue as the bottleneck of the
// short-K GEMMs -- 7 750 clk per 128x256 tile against 3 500 for loads + MMA -- with ~970 clk per pass spent by the epilogue
// leader ISSUING the four 5-D TMA stores while the other 255 epilogue threads waited at a barrier, and three bar.sync per
// pass; now the epilogue warps only compute and stage, hand a full staging buffer to the store thread through an mbarrier
// and continue with the other buffer), warps 4-11 epilogue: warp w owns TMEM lanes 32*(w%4)..+31 (= tile rows) and every other 32-column chunk
// (the GEGLU / residual epilogues are instruction-bound with one warp per quadrant).
#pragma once
#include "common.cuh"
#include "tapgemm.cuh"

// Instrumented build (tools/build_variant.py -DSTAR_GEMM_TRACE=1):
//   STAR_GEMM_TRACE 1: CTA 0 records clock64() timestamps of its producer / MMA / epilogue roles per tile into g_tg2_trace
//                     (tools/gemm_trace.py reads it back through star_debug_read_trace); never set in the shipped library.
#ifndef STAR_GEMM_TRACE
#define STAR_GEMM_TRACE 0
#endif

namespace star {

#if STAR_GEMM_TRACE
__device__ long long g_tg2_trace[3][4096];        // [role][slot]: role 0 producer, 1 MMA, 2 epilogue (warp 4 lane 0)
__device__ int g_tg2_trace_n[3];
STAR_DEVINL void tg2_trace(int role, int event) {
    if (blockIdx.x != 0) return;
    const int i = g_tg2_trace_n[role];
    if (i + 1 < 4096) {
        g_tg2_trace[role][i] = event;
        g_tg2_trace[role][i + 1] = clock64();
        g_tg2_trace_n[role] = i + 2;
    }
}
#define TG2_TRACE(role, event) tg2_trace(role, event)
#else
#define TG2_TRACE(role, event)
#endif

constexpr int TG2_THREADS = 384;      // warps 0-3: TMA, MMA, 2 idle; warps 4-11: epilogue (two warps per TMEM lane quadrant)
constexpr int TG2_MAX_STAGES = 6;

template <int BN>
struct TapGemm2Smem {
    static constexpr int A_BYTES = TG_BM * TG_BK * 2;
    static constexpr int B_BYTES = BN * TG_BK * 2;
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    // BN = 256 (48 KB stages): the staging buffer holds 128 output columns and the epilogue makes two passes over it,
    // and the residual is read straight from global memory -- that leaves room for 4 operand stages.
    static constexpr int OUT_COLS = BN > 160 ? 128 : BN;
    static constexpr bool RES_TMA = BN <= 160;
    static constexpr int OUT_BYTES = TG_BM * OUT_COLS * 2;            // OUT_COLS/32 sub-tiles of [128 rows x 64 B]
    static constexpr int BUDGET = 232448 - 1024 - 256;                // 227 KB minus alignment slack and barriers
    // as many operand stages as fit beside the staging buffer(s) (and the residual buffer when it is TMA-prefetched)
    static constexpr int stages(bool res_tma, bool dbuf = false) {
        int n = (BUDGET - OUT_BYTES * ((dbuf ? 2 : 1) + (res_tma ? 1 : 0))) / STAGE_BYTES;
        return n > TG2_MAX_STAGES ? TG2_MAX_STAGES : n;
    }
    static constexpr int total(bool res_tma, bool dbuf = false) {
        return stages(res_tma, dbuf) * STAGE_BYTES + OUT_BYTES * ((dbuf ? 2 : 1) + (res_tma ? 1 : 0)) + 256 + 1024;
    }
};

STAR_DEVINL void tma_store_5d(const CUtensorMap* m, const void* src, int c0, int c1, int c2, int c3, int c4) {
    asm volatile("cp.async.bulk.tensor.5d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];"
                 ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
                 : "memory");
}
STAR_DEVINL void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
STAR_DEVINL void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
STAR_DEVINL void tma_store_wait_read_but_one() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
STAR_DEVINL void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
STAR_DEVINL void epi_bar_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

struct TapGemm2Extra {
    int num_tiles;        // m_tiles * n_tiles
    int n_tiles;
    int stages;           // operand ring depth (depends on BN, the residual buffer and the staging depth)
    int dbuf;             // 1: two output staging buffers -- the TMA-store drain of pass i overlaps the arithmetic of pass i+1
                          //    (attribution, profiles/r02_kbench_gemm_attribution.log: with one buffer the short-K GEMMs lose
                          //    25-30 % to the serialised drain)
};

// EPI selects a compile-time specialisation of the epilogue (the role timeline showed the generic epilogue -- ~1 500 SASS
// instructions of run-time-flag paths per 32-column chunk -- as the limiter of the short-K GEMMs):
//   0 generic (every flag / pointer combination)      1 plain: (+bias) only
//   2 (+bias) + TMA-prefetched residual                3 GEGLU (+bias)
enum { TG2_EPI_GENERIC = 0, TG2_EPI_PLAIN = 1, TG2_EPI_RES = 2, TG2_EPI_GEGLU = 3 };

template <int BN, int EPI = TG2_EPI_GENERIC>
__global__ void __launch_bounds__(TG2_THREADS, 1)
tapgemm2_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_w,
                const __grid_constant__ CUtensorMap tmap_out, const __grid_constant__ CUtensorMap tmap_res,
                const __grid_constant__ TapGemmParams p, const __grid_constant__ TapGemm2Extra ex) {
    using SM = TapGemm2Smem<BN>;
    constexpr uint32_t ACC_STRIDE = (BN <= 128) ? 128 : 256;          // TMEM columns between the two accumulators
    constexpr uint32_t TMEM_COLS = 2 * ACC_STRIDE;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int NS = ex.stages;
    const int OFF_OUT = NS * SM::STAGE_BYTES;
    const int OFF_RES = OFF_OUT + SM::OUT_BYTES * (ex.dbuf ? 2 : 1);
    constexpr bool GEN = EPI == TG2_EPI_GENERIC;
    // residual tile prefetched by TMA (else: direct loads)
    const bool res_tma = EPI == TG2_EPI_RES ? true : (GEN && SM::RES_TMA && p.residual != nullptr);
    const int OFF_BAR = OFF_RES + (res_tma ? SM::OUT_BYTES : 0);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
    uint64_t* empty_bar = full_bar + TG2_MAX_STAGES;
    uint64_t* acc_full = empty_bar + TG2_MAX_STAGES; // 2
    uint64_t* acc_empty = acc_full + 2;              // 2
    uint64_t* res_full = acc_empty + 2;              // 1
    uint64_t* res_empty = res_full + 1;              // 1
    uint64_t* stage_full = res_empty + 1;            // 2   epilogue warps -> store thread: staging buffer b holds a finished pass
    uint64_t* stage_empty = stage_full + 2;          // 2   store thread -> epilogue warps: the TMA stores of buffer b have read it
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(stage_empty + 2);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const bool geglu = EPI == TG2_EPI_GEGLU ? true : (GEN && (p.flags & TG_GEGLU) != 0);
    const bool has_res = EPI == TG2_EPI_RES ? true : (GEN && p.residual != nullptr);
    const bool has_rowvec = GEN && p.rowvec != nullptr;
    const bool has_colscale = GEN && p.colscale != nullptr;
    const bool act_tanh = GEN && (p.flags & TG_GELU_TANH) != 0;
    const bool act_erf = GEN && (p.flags & TG_GELU_ERF) != 0;
    const bool act_silu = GEN && (p.flags & TG_SILU_OUT) != 0;
    const int n_per_tile = geglu ? BN / 2 : BN;
    const int total_iters = p.ntaps * p.k_chunks;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmap_a);
        tma_prefetch_desc(&tmap_w);
        tma_prefetch_desc(&tmap_out);
        if (has_res) tma_prefetch_desc(&tmap_res);
    }
    if (warp == 1) {
        if (lane == 0) {
            for (int s = 0; s < NS; ++s) {
                mbar_init(&full_bar[s], 1);
                mbar_init(&empty_bar[s], 1);
            }
            for (int b = 0; b < 2; ++b) {
                mbar_init(&acc_full[b], 1);
                mbar_init(&acc_empty[b], 256);
            }
            mbar_init(res_full, 1);
            mbar_init(res_empty, 256);
            for (int b = 0; b < 2; ++b) {
                mbar_init(&stage_full[b], 256);
                mbar_init(&stage_empty[b], 1);
            }
            fence_barrier_init();
        }
        __syncwarp();
        tmem_alloc<TMEM_COLS>(tmem_slot);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    auto tile_origin = [&](int tile, int* org, int& n_tile) {
        n_tile = tile % ex.n_tiles;
        int m_tile = tile / ex.n_tiles;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            org[i] = (m_tile % p.tiles[i]) * p.box[i];
            m_tile /= p.tiles[i];
        }
    };

    if (warp == 0) {
        // ------------------------------------------------ TMA producer
        if (lane == 0) {
            const uint32_t tx = (uint32_t)p.box_rows * 128u + (uint32_t)SM::B_BYTES;
            int s = 0, local = 0;
            uint32_t ph = 0;                              // ring phase (no runtime div/mod in the issue loops)
            for (int tile = blockIdx.x; tile < ex.num_tiles; tile += gridDim.x, ++local) {
                int org[4], n_tile;
                tile_origin(tile, org, n_tile);
                TG2_TRACE(0, 1);                                   // producer: tile start
                for (int t = 0; t < p.ntaps; ++t) {
                    const int c1 = org[0] + p.tap[t][0], c2 = org[1] + p.tap[t][1];
                    const int c3 = org[2] + p.tap[t][2], c4 = org[3] + p.tap[t][3];
                    for (int kc = 0; kc < p.k_chunks; ++kc) {
                        mbar_wait(&empty_bar[s], ph ^ 1);
                        uint8_t* sa = smem + s * SM::STAGE_BYTES;
                        uint8_t* sb = sa + SM::A_BYTES;
                        mbar_expect_tx(&full_bar[s], tx);
                        tma_load_5d(sa, &tmap_a, &full_bar[s], kc * TG_BK, c1, c2, c3, c4);
                        const int kw = t * p.K + kc * TG_BK;
                        if (!geglu) {
                            tma_load_2d(sb, &tmap_w, &full_bar[s], kw, n_tile * BN);
                        } else {
                            tma_load_2d(sb, &tmap_w, &full_bar[s], kw, n_tile * (BN / 2));
                            tma_load_2d(sb + (BN / 2) * 128, &tmap_w, &full_bar[s], kw, p.N + n_tile * (BN / 2));
                        }
                        if (++s == NS) { s = 0; ph ^= 1; }
                    }
                }
                TG2_TRACE(0, 2);                                   // producer: all operand loads of the tile issued
                if (res_tma) {
                    // residual tile of THIS output tile, issued after its operand loads so that waiting for the
                    // previous epilogue to release the buffer never delays the operand prefetch
                    const int n_base = n_tile * n_per_tile;
                    int nsub = (p.N - n_base + 31) / 32;
                    nsub = nsub < n_per_tile / 32 ? nsub : n_per_tile / 32;
                    mbar_wait(res_empty, (local & 1) ^ 1);
                    mbar_expect_tx(res_full, (uint32_t)p.box_rows * 64u * nsub);
#pragma unroll 1
                    for (int sb = 0; sb < nsub; ++sb)
                        tma_load_5d(smem + OFF_RES + sb * 8192, &tmap_res, res_full, n_base + sb * 32, org[0], org[1],
                                    org[2], org[3]);
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------ MMA issuer
        if (lane == 0) {
            constexpr uint32_t idesc = umma_idesc_f16(TG_BM, BN, 0, 0);
            // The single issuing thread is on the critical path (ncu: tensor pipe 40 % busy with L2 at 50 % when each
            // k-step rebuilt two 64-bit descriptors): descriptors are formed once, a stage / k-step is a 64-bit add.
            const uint64_t desc_a0 = umma_desc_sw128(smem_u32(smem), 16, 1024);
            const uint64_t desc_b0 = umma_desc_sw128(smem_u32(smem) + SM::A_BYTES, 16, 1024);
            constexpr uint64_t STAGE_INC = (uint64_t)(SM::STAGE_BYTES >> 4);
            int s = 0, local = 0;
            uint32_t ph = 0;
            for (int tile = blockIdx.x; tile < ex.num_tiles; tile += gridDim.x, ++local) {
                const int buf = local & 1;
                TG2_TRACE(1, 1);                                   // MMA: waiting for the accumulator
                mbar_wait(&acc_empty[buf], ((local >> 1) & 1) ^ 1);
                tc_fence_after();
                TG2_TRACE(1, 2);                                   // MMA: accumulator free
                const uint32_t acc = tmem_base + buf * ACC_STRIDE;
                for (int i = 0; i < total_iters; ++i) {
                    mbar_wait(&full_bar[s], ph);
                    tc_fence_after();
                    const uint64_t da = desc_a0 + STAGE_INC * (uint64_t)s;
                    const uint64_t db = desc_b0 + STAGE_INC * (uint64_t)s;
                    umma_f16_ss(acc, da, db, idesc, i > 0 ? 1u : 0u);
                    umma_f16_ss(acc, da + 2, db + 2, idesc, 1u);
                    umma_f16_ss(acc, da + 4, db + 4, idesc, 1u);
                    umma_f16_ss(acc, da + 6, db + 6, idesc, 1u);
                    umma_commit(&empty_bar[s]);
                    if (++s == NS) { s = 0; ph ^= 1; }
                }
                umma_commit(&acc_full[buf]);
                TG2_TRACE(1, 3);                                   // MMA: last instruction of the tile issued
            }
        }
    } else if (warp == 3) {
        // ------------------------------------------------ TMA-store thread: drains finished staging buffers
        if (lane == 0) {
            constexpr int PASS_COLS = SM::OUT_COLS;
            int pc = 0;                                    // passes so far (same sequence as the epilogue warps)
            for (int tile = blockIdx.x; tile < ex.num_tiles; tile += gridDim.x) {
                int org[4], n_tile;
                tile_origin(tile, org, n_tile);
                const int n_base = n_tile * n_per_tile;
                for (int pass0 = 0; pass0 < n_per_tile; pass0 += PASS_COLS, ++pc) {
                    const int ob = ex.dbuf ? (pc & 1) : 0;
                    const int use = ex.dbuf ? (pc >> 1) : pc;          // how often this buffer has been used before
                    const int pass_end = (pass0 + PASS_COLS < n_per_tile) ? pass0 + PASS_COLS : n_per_tile;
                    mbar_wait(&stage_full[ob], use & 1);
#pragma unroll 1
                    for (int sb = 0; sb < (pass_end - pass0) / 32; ++sb) {
                        if (n_base + pass0 + sb * 32 < p.N)
                            tma_store_5d(&tmap_out, smem + OFF_OUT + ob * SM::OUT_BYTES + sb * 8192, n_base + pass0 + sb * 32,
                                         org[0], org[1], org[2], org[3]);
                    }
                    tma_store_commit();
                    tma_store_wait_read();                 // with two buffers the epilogue warps fill the other one meanwhile
                    mbar_arrive(&stage_empty[ob]);
                }
            }
            tma_store_wait_all();
        }
    } else if (warp >= 4) {
        // ------------------------------------------------ epilogue warps 4..11
        const int q = warp & 3;
        const int ehalf = (warp - 4) >> 2;                  // this warp handles 32-column chunks with (chunk & 1) == ehalf
        const int r = q * 32 + lane;
        const uint32_t lane_off = (uint32_t)(q * 32) << 16;
        const int swz = (r >> 1) & 3;                       // SWIZZLE_64B: 16-byte chunk index ^= (row / 2) % 4
        uint8_t* out_row0 = smem + OFF_OUT + r * 64;
        const uint8_t* res_row = smem + OFF_RES + r * 64;
        const bool leader = (threadIdx.x == 4 * 32);
        int local = 0;
        int pass_ctr = 0;
        for (int tile = blockIdx.x; tile < ex.num_tiles; tile += gridDim.x, ++local) {
            int org[4], n_tile;
            tile_origin(tile, org, n_tile);
            const int buf = local & 1;
            const int n_base = n_tile * n_per_tile;
            // global output row of this tile row (clamped to the tensor for clipped rows): time-embedding row
            // (unet_v2v.py:684; rows of one tile may belong to different clips) and direct residual loads
            const __half* rv_row = nullptr;
            const __half* res_g = nullptr;
            if (has_rowvec || (has_res && !res_tma)) {
                int rr = r;
                long long orow = 0, mul = 1;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int l = rr % p.box[i];
                    rr /= p.box[i];
                    int g = org[i] + l;
                    g = g < p.on[i] ? g : p.on[i] - 1;
                    orow += (long long)g * mul;
                    mul *= p.on[i];
                }
                if (has_rowvec) rv_row = p.rowvec + (orow / p.rowvec_div) * p.rowvec_ld;
                if (has_res && !res_tma) res_g = p.residual + orow * p.res_ld;
            }
            if (leader) TG2_TRACE(2, 1);                           // epilogue: waiting for acc_full
            mbar_wait(&acc_full[buf], (local >> 1) & 1);
            tc_fence_after();
            if (leader) TG2_TRACE(2, 2);                           // epilogue: accumulator complete
            if (res_tma) mbar_wait(res_full, local & 1);
            const uint32_t t_row = tmem_base + buf * ACC_STRIDE + lane_off;
            const int last_c0 = ((n_per_tile / 32 - 1 - ehalf) & ~1) * 32 + ehalf * 32;   // last chunk of this warp
            constexpr int PASS_COLS = SM::OUT_COLS;
#pragma unroll 1
            for (int pass0 = 0; pass0 < n_per_tile; pass0 += PASS_COLS) {
            // the TMA stores that last used this staging buffer must have finished reading it (store thread -> stage_empty)
            const int ob = ex.dbuf ? (pass_ctr & 1) : 0;
            const int use = ex.dbuf ? (pass_ctr >> 1) : pass_ctr;
            ++pass_ctr;
            uint8_t* out_row = out_row0 + ob * SM::OUT_BYTES;
            if (leader) TG2_TRACE(2, 3);                           // pass: before the staging-buffer wait
            mbar_wait(&stage_empty[ob], (use & 1) ^ 1);
            if (leader) TG2_TRACE(2, 4);                           // pass: staging buffer free
            const int pass_end = (pass0 + PASS_COLS < n_per_tile) ? pass0 + PASS_COLS : n_per_tile;
#pragma unroll 1
            for (int c0 = pass0 + ehalf * 32; c0 < pass_end; c0 += 64) {
                uint32_t v[32];
                float f[32];
                tmem_ld32(t_row + c0, v);
                const int n0 = n_base + c0;
                if (geglu) {
                    uint32_t g[32];
                    tmem_ld32(t_row + (BN / 2) + c0, g);
                    tmem_ld_wait();
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        float bv[8], bg[8];
                        const bool inb = (n0 + u * 8 + 8 <= p.N) && p.bias;
                        if (inb) {
                            unpack8h(__ldg(reinterpret_cast<const uint4*>(p.bias + n0 + u * 8)), bv);
                            unpack8h(__ldg(reinterpret_cast<const uint4*>(p.bias + p.N + n0 + u * 8)), bg);
                        }
#pragma unroll
                        for (int e = 0; e < 8; ++e) {
                            float xv = __uint_as_float(v[u * 8 + e]), gv = __uint_as_float(g[u * 8 + e]);
                            if (inb) { xv += bv[e]; gv += bg[e]; }
                            f[u * 8 + e] = xv * gelu_erf_f(gv);
                        }
                    }
                } else {
                    tmem_ld_wait();
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        float bv[8];
                        const bool inb = (n0 + u * 8 + 8 <= p.N) && p.bias;
                        if (inb) unpack8h(__ldg(reinterpret_cast<const uint4*>(p.bias + n0 + u * 8)), bv);
#pragma unroll
                        for (int e = 0; e < 8; ++e) f[u * 8 + e] = __uint_as_float(v[u * 8 + e]) + (inb ? bv[e] : 0.f);
                    }
                }
                if (c0 == last_c0) {                         // last TMEM read of this warp for this accumulator
                    tc_fence_before();
                    mbar_arrive(&acc_empty[buf]);
                }
                if (act_tanh) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) f[j] = gelu_tanh_f(f[j]);
                }
                if (act_erf) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) f[j] = gelu_erf_f(f[j]);
                }
                if (has_colscale) {
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        if (n0 + u * 8 + 8 <= p.N) {
                            float cs[8];
                            unpack8h(__ldg(reinterpret_cast<const uint4*>(p.colscale + n0 + u * 8)), cs);
#pragma unroll
                            for (int e = 0; e < 8; ++e) f[u * 8 + e] *= cs[e];
                        }
                    }
                }
                if (has_rowvec && rv_row) {
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        if (n0 + u * 8 + 8 <= p.N) {
                            float tv[8];
                            unpack8h(__ldg(reinterpret_cast<const uint4*>(rv_row + n0 + u * 8)), tv);
#pragma unroll
                            for (int e = 0; e < 8; ++e) f[u * 8 + e] += tv[e];
                        }
                    }
                }
                const int sub = (c0 - pass0) >> 5;
                if (res_tma) {
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        float rv[8];
                        unpack8h(*reinterpret_cast<const uint4*>(res_row + sub * 8192 + ((u ^ swz) * 16)), rv);
#pragma unroll
                        for (int e = 0; e < 8; ++e) f[u * 8 + e] += rv[e];
                    }
                } else if (GEN && res_g) {
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        if (n0 + u * 8 + 8 <= p.N) {
                            float rv[8];
                            unpack8h(__ldg(reinterpret_cast<const uint4*>(res_g + n0 + u * 8)), rv);
#pragma unroll
                            for (int e = 0; e < 8; ++e) f[u * 8 + e] += rv[e];
                        }
                    }
                }
                if (act_silu) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) f[j] = silu_f(f[j]);
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    uint4 o;
                    o.x = pack_half2(f[u * 8 + 0], f[u * 8 + 1]);
                    o.y = pack_half2(f[u * 8 + 2], f[u * 8 + 3]);
                    o.z = pack_half2(f[u * 8 + 4], f[u * 8 + 5]);
                    o.w = pack_half2(f[u * 8 + 6], f[u * 8 + 7]);
                    *reinterpret_cast<uint4*>(out_row + sub * 8192 + ((u ^ swz) * 16)) = o;
                }
            }
            if (res_tma && pass_end == n_per_tile) mbar_arrive(res_empty);
            if (leader) TG2_TRACE(2, 6);                           // pass: this warp's chunks computed and staged
            fence_proxy_async_smem();                              // generic-proxy writes -> visible to the TMA store (async proxy)
            mbar_arrive(&stage_full[ob]);
            }
        }
    }
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc<TMEM_COLS>(tmem_base);
    }
}

}  // namespace star
