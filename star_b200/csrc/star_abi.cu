// star_b200 / csrc / star_abi.cu -- host side of libstar_sm100.so (C ABI in include/star_sm100.h)
#include <cuda.h>
#include <cudaTypedefs.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

#include "../../include/star_sm100.h"
#include "attn.cuh"
#include "attn4.cuh"
#include "rowops.cuh"
#include "tattn2.cuh"
#include "tapgemm.cuh"
#include "tapgemm2.cuh"

using namespace star;

namespace {

thread_local std::string g_err;
PFN_cuTensorMapEncodeTiled_v12000 g_encode = nullptr;
constexpr int STAR_MAX_DEVICES = 64;
int g_sms[STAR_MAX_DEVICES] = {0};            // SM count per initialised device (0 = star_init not called for it)
// Tile-shape rules of the tap-GEMM dispatch (measured: profiles/r01_kbench_wide_tiles.log); constants, not switches.
constexpr int kWideWastePct = 10;             // largest padding (percent of N) accepted for the 128x256 tiles ...
constexpr int kWideWasteLongKPct = 25;        // ... and for reductions >= 1920 (N = 640 as 3 x 256: +16 % on the 640-channel convs)
constexpr int kWideMinK = 256;                // smallest reduction length that takes the 128x256 tiles
constexpr int kDbufMaxK = 700;                // 128x256-tile GEMMs with reductions up to this length use two output staging buffers
                                              // (A/B: profiles/r02_kbench_gemm_dbuf_ab.log -- qkv -5 %, 512->1536 -9 %, longer K / narrower tiles lose)
std::atomic<long long> g_launches{0};

// SM count of the CURRENT device (kernels are launched on the caller's current device / stream)
inline int num_sms() {
    int dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess && dev >= 0 && dev < STAR_MAX_DEVICES && g_sms[dev] > 0) return g_sms[dev];
    return 148;
}

int fail(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return 1;
}

#define STAR_CHECK_INIT()                                                                                        \
    do {                                                                                                         \
        int dev_ = -1;                                                                                           \
        if (!g_encode || cudaGetDevice(&dev_) != cudaSuccess || dev_ < 0 || dev_ >= STAR_MAX_DEVICES || !g_sms[dev_]) \
            return fail("star_init(%d) has not been called for the current device (or failed)", dev_);           \
    } while (0)
#define STAR_CUDA(x)                                                                        \
    do {                                                                                    \
        cudaError_t e_ = (x);                                                               \
        if (e_ != cudaSuccess) return fail("%s failed: %s", #x, cudaGetErrorString(e_));    \
    } while (0)
#define STAR_LAUNCH_CHECK(name)                                                             \
    do {                                                                                    \
        g_launches.fetch_add(1, std::memory_order_relaxed);                                 \
        cudaError_t e_ = cudaGetLastError();                                                \
        if (e_ != cudaSuccess) return fail("launch %s failed: %s", name, cudaGetErrorString(e_)); \
    } while (0)

// rank-`rank` fp16 tensor map, dims[0] innermost (contiguous), strides in ELEMENTS for dims 1..rank-1
int make_tmap(CUtensorMap* m, const void* base, int rank, const unsigned long long* dims,
              const unsigned long long* strides_elems, const unsigned* box,
              CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
    cuuint64_t gdim[5], gstr[4];
    cuuint32_t bx[5], es[5];
    for (int i = 0; i < rank; ++i) {
        gdim[i] = dims[i];
        bx[i] = box[i];
        es[i] = 1;
        if (i > 0) {
            gstr[i - 1] = strides_elems[i] * 2ull;
            if (gstr[i - 1] % 16) return fail("tensor map stride %llu B of dim %d is not a multiple of 16", (unsigned long long)gstr[i - 1], i);
        }
        if (box[i] == 0 || box[i] > 256) return fail("tensor map box[%d]=%u out of range", i, box[i]);
    }
    if (reinterpret_cast<uintptr_t>(base) % 16) return fail("tensor map base not 16-byte aligned");
    CUresult r = g_encode(m, STAR_TMAP_DTYPE, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstr, bx, es,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    return 0;
}

inline int grid_for(long long n, int block, int cap_mult = 32) {
    long long g = (n + block - 1) / block;
    return (int)std::max(1ll, std::min(g, (long long)num_sms() * cap_mult));
}

// ------------------------------------------------------------------ tap-GEMM launcher
struct TapDesc {
    const void* A;
    unsigned long long adim[5];      // (C, n1..n4) of the input view
    unsigned long long astr[5];      // element strides of dims 1..4 (astr[0] unused)
    int on[4];                       // output extents
    int box[4];
    int ntaps;
    int tap[TG_MAX_TAPS][4];
    int K, N, flags;
    const void *W, *bias, *rowvec, *residual, *colscale;
    long long rowvec_div, ldrowvec, ldres, ldo;
    void* out;
};

// Shared by both tap-GEMM kernels: the kernel parameters, the number of M tiles, and the tensor maps of the input view (A)
// and of the weights (W, BN rows per box; GEGLU: BN / 2 value rows and BN / 2 gate rows).  `name` prefixes the error message.
template <int BN>
int tapgemm_setup(const TapDesc& d, const char* name, TapGemmParams& p, long long& m_tiles, CUtensorMap& ta,
                  CUtensorMap& tw) {
    memset(&p, 0, sizeof(p));
    m_tiles = 1;
    int box_rows = 1;
    for (int i = 0; i < 4; ++i) {
        p.on[i] = d.on[i];
        p.box[i] = d.box[i];
        p.tiles[i] = (d.on[i] + d.box[i] - 1) / d.box[i];
        m_tiles *= p.tiles[i];
        box_rows *= d.box[i];
    }
    if (box_rows > TG_BM) return fail("%s: box has %d rows (> %d)", name, box_rows, TG_BM);
    p.box_rows = box_rows;
    p.ntaps = d.ntaps;
    memcpy(p.tap, d.tap, sizeof(p.tap));
    p.K = d.K;
    p.k_chunks = (d.K + TG_BK - 1) / TG_BK;
    p.N = d.N;
    p.flags = d.flags;
    p.bias = (const __half*)d.bias;
    p.rowvec = (const __half*)d.rowvec;
    p.rowvec_div = (int)std::max(1ll, d.rowvec_div);
    p.rowvec_ld = d.ldrowvec > 0 ? d.ldrowvec : d.N;
    p.residual = (const __half*)d.residual;
    p.colscale = (const __half*)d.colscale;
    p.res_ld = d.ldres;
    p.out = (__half*)d.out;
    p.out_ld = d.ldo;

    const bool geglu = d.flags & TG_GEGLU;
    unsigned abox[5] = {TG_BK, (unsigned)d.box[0], (unsigned)d.box[1], (unsigned)d.box[2], (unsigned)d.box[3]};
    if (make_tmap(&ta, d.A, 5, d.adim, d.astr, abox)) return 1;
    const unsigned long long wrows = geglu ? 2ull * d.N : (unsigned long long)d.N;
    unsigned long long wdim[2] = {(unsigned long long)d.ntaps * d.K, wrows};
    unsigned long long wstr[2] = {1, (unsigned long long)d.ntaps * d.K};
    unsigned wbox[2] = {TG_BK, (unsigned)(geglu ? BN / 2 : BN)};
    return make_tmap(&tw, d.W, 2, wdim, wstr, wbox);
}

template <int BN>
int launch_tapgemm_bn(const TapDesc& d, cudaStream_t st) {
    TapGemmParams p;
    long long m_tiles;
    CUtensorMap ta, tw;
    if (tapgemm_setup<BN>(d, "tapgemm", p, m_tiles, ta, tw)) return 1;
    const bool geglu = d.flags & TG_GEGLU;
    if (geglu && BN != 128) return fail("tapgemm: GEGLU requires BN=128");
    if (geglu && (d.N % 64)) return fail("tapgemm: GEGLU requires N %% 64 == 0 (N=%d)", d.N);
    if (m_tiles > 65535) return fail("tapgemm: %lld M tiles exceed grid.y", m_tiles);

    const int n_per_tile = geglu ? BN / 2 : BN;
    dim3 grid((d.N + n_per_tile - 1) / n_per_tile, (unsigned)m_tiles, 1);
    tapgemm_kernel<BN><<<grid, TG_THREADS, TapGemmSmem<BN>::TOTAL, st>>>(ta, tw, p);
    STAR_LAUNCH_CHECK("tapgemm");
    return 0;
}

template <int BN>
int launch_tapgemm2_bn(const TapDesc& d, cudaStream_t st) {
    TapGemmParams p;
    long long m_tiles;
    CUtensorMap ta, tw, to, tr;
    if (tapgemm_setup<BN>(d, "tapgemm2", p, m_tiles, ta, tw)) return 1;
    const bool geglu = d.flags & TG_GEGLU;
    const int n_per_tile = geglu ? BN / 2 : BN;
    TapGemm2Extra ex;
    ex.n_tiles = (d.N + n_per_tile - 1) / n_per_tile;
    const long long total = m_tiles * ex.n_tiles;
    if (total > 0x7fffffffll) return fail("tapgemm2: too many tiles");
    ex.num_tiles = (int)total;

    // output / residual: (N, n1..n4) with row pitch ld; 32-column boxes, SWIZZLE_64B staging tiles
    unsigned obox[5] = {32, (unsigned)d.box[0], (unsigned)d.box[1], (unsigned)d.box[2], (unsigned)d.box[3]};
    unsigned long long odim[5] = {(unsigned long long)d.N, (unsigned long long)d.on[0], (unsigned long long)d.on[1],
                                  (unsigned long long)d.on[2], (unsigned long long)d.on[3]};
    auto strides = [&](long long ld, unsigned long long* s) {
        s[0] = 1;
        s[1] = (unsigned long long)ld;
        s[2] = s[1] * d.on[0];
        s[3] = s[2] * d.on[1];
        s[4] = s[3] * d.on[2];
    };
    unsigned long long ostr[5], rstr[5];
    strides(d.ldo, ostr);
    if (make_tmap(&to, d.out, 5, odim, ostr, obox, CU_TENSOR_MAP_SWIZZLE_64B)) return 1;
    // Output staging depth.  Short reductions are epilogue-bound (the main loop alone runs at 75-82 % of peak, the serialised
    // store drain costs 25-30 %: profiles/r02_kbench_gemm_attribution.log) -> two staging buffers, one operand stage fewer.
    ex.dbuf = ((long long)d.ntaps * d.K <= kDbufMaxK) ? 1 : 0;
    const bool res_tma = d.residual && TapGemm2Smem<BN>::RES_TMA;
    if (ex.dbuf && TapGemm2Smem<BN>::stages(res_tma, true) < 3) ex.dbuf = 0;       // BN = 160 + residual: no room for a second buffer
    if (res_tma) {
        strides(d.ldres, rstr);
        if (make_tmap(&tr, d.residual, 5, odim, rstr, obox, CU_TENSOR_MAP_SWIZZLE_64B)) return 1;
    } else {
        tr = to;
    }
    const int grid = (int)std::min<long long>(total, num_sms());
    ex.stages = TapGemm2Smem<BN>::stages(res_tma, ex.dbuf != 0);
    const size_t smem = TapGemm2Smem<BN>::total(res_tma, ex.dbuf != 0);
    // compile-time specialised epilogues for the three shapes that carry ~all of the linear / conv time
    const bool extras = d.rowvec || d.colscale || (d.flags & (TG_GELU_TANH | TG_GELU_ERF | TG_SILU_OUT));
    bool launched = false;
    if (geglu && !d.residual && !extras) {
        if constexpr (BN != 160) {
            tapgemm2_kernel<BN, TG2_EPI_GEGLU><<<grid, TG2_THREADS, smem, st>>>(ta, tw, to, tr, p, ex);
            launched = true;
        }
    } else if (!geglu && !d.residual && !extras) {
        tapgemm2_kernel<BN, TG2_EPI_PLAIN><<<grid, TG2_THREADS, smem, st>>>(ta, tw, to, tr, p, ex);
        launched = true;
    } else if (!geglu && res_tma && !extras) {
        if constexpr (TapGemm2Smem<BN>::RES_TMA) {
            tapgemm2_kernel<BN, TG2_EPI_RES><<<grid, TG2_THREADS, smem, st>>>(ta, tw, to, tr, p, ex);
            launched = true;
        }
    }
    if (!launched) tapgemm2_kernel<BN, TG2_EPI_GENERIC><<<grid, TG2_THREADS, smem, st>>>(ta, tw, to, tr, p, ex);
    STAR_LAUNCH_CHECK("tapgemm2");
    return 0;
}

int launch_tapgemm(const TapDesc& d, cudaStream_t st) {
    const bool geglu = d.flags & TG_GEGLU;
    const bool aligned = (d.N % 32 == 0) && (d.ldo % 8 == 0) && (reinterpret_cast<uintptr_t>(d.out) % 16 == 0) &&
                         (!d.residual || ((d.ldres % 8 == 0) && (reinterpret_cast<uintptr_t>(d.residual) % 16 == 0))) &&
                         (!geglu || d.N % 64 == 0);
    // Non-persistent kernel (2 CTAs/SM, two interleaved MMA streams) is measurably faster for the long-reduction,
    // wide-N convolutions (profiles/r01_kbench_ab_experiments.txt); the persistent one wins everywhere else.
    const bool v2_only = d.colscale != nullptr || (d.flags & (TG_GELU_TANH | TG_GELU_ERF));
    if (v2_only && !aligned) return fail("tapgemm: colscale / GELU epilogues need N %% 32 == 0 and 16-byte aligned rows");
    const bool long_k = ((long long)d.ntaps * d.K >= 3840) && (d.N % 128 == 0) && !geglu && !v2_only;
    // 128x256 tiles (4 x 48 KB stages, two-pass epilogue): 25 % less L2->SM operand traffic per flop and N = 256 MMAs
    // (137 clk per instruction against a 128 clk floor; N = 128 retires at 73 against 64: profiles/r01_micro_mma_rate.log)
    // Used when the padded width wastes <= 10 % (<= 25 % for long reductions, where the tile-shape gain outweighs it:
    // profiles/r01_kbench_wide_tiles.log) (N = 960, 1280, 1920, 2560, 3840, ...; GEGLU: 128 outputs per tile).
    const int wide_n = geglu ? 128 : 256;
    const long long padded = ((long long)d.N + wide_n - 1) / wide_n * wide_n;
    const long long red = (long long)d.ntaps * d.K;
    const bool wide = aligned && red >= kWideMinK &&
                      padded * 100 <= (long long)d.N * (100 + (red >= 1920 ? kWideWasteLongKPct : kWideWastePct));
    if (wide) return launch_tapgemm2_bn<256>(d, st);
    const bool n160 = !geglu && d.N % 160 == 0 && d.N % 128 != 0;
    if (aligned && !long_k) return n160 ? launch_tapgemm2_bn<160>(d, st) : launch_tapgemm2_bn<128>(d, st);
    return n160 ? launch_tapgemm_bn<160>(d, st) : launch_tapgemm_bn<128>(d, st);
}

void best_box_2d(int H, int W, int* th, int* tw) {
    long long best = -1;
    for (int w = 1; w <= std::min(W, 128); ++w) {
        int h = std::min(H, 128 / w);
        if (h < 1) continue;
        long long tiles = (long long)((W + w - 1) / w) * ((H + h - 1) / h);
        if (best < 0 || tiles < best || (tiles == best && w > *tw)) {
            best = tiles;
            *th = h;
            *tw = w;
        }
    }
}

}  // namespace

extern "C" {

#ifdef STAR_BF16
int star_version(void) { return 101; }     /* odd: bf16 build */
#else
int star_version(void) { return 100; }
#endif
const char* star_last_error(void) { return g_err.c_str(); }
long long star_launch_count(void) { return g_launches.load(); }

// Per-device initialisation: checks the architecture, records the SM count and raises the dynamic shared-memory limit of
// every kernel ON THAT DEVICE (function attributes are per device).  The caller's current device is restored.
static int star_init_on_current(int device) {
    cudaDeviceProp prop;
    STAR_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail("libstar_sm100 needs an sm_100 device, found sm_%d%d", prop.major, prop.minor);
    if (!g_encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qr;
        STAR_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qr));
        if (!fn || qr != cudaDriverEntryPointSuccess) return fail("cuTensorMapEncodeTiled not available from the driver");
        g_encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
    }
#define STAR_SMEM_ATTR(kernel, bytes) STAR_CUDA((cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes))))
    STAR_SMEM_ATTR(tapgemm_kernel<128>, TapGemmSmem<128>::TOTAL);
    STAR_SMEM_ATTR(tapgemm_kernel<160>, TapGemmSmem<160>::TOTAL);
    STAR_SMEM_ATTR((tapgemm2_kernel<128, TG2_EPI_GENERIC>), 232448);
    STAR_SMEM_ATTR((tapgemm2_kernel<160, TG2_EPI_GENERIC>), 232448);
    STAR_SMEM_ATTR((tapgemm2_kernel<256, TG2_EPI_GENERIC>), 232448);
    STAR_SMEM_ATTR((tapgemm2_kernel<128, TG2_EPI_PLAIN>), 232448);
    STAR_SMEM_ATTR((tapgemm2_kernel<160, TG2_EPI_PLAIN>), 232448);
    STAR_SMEM_ATTR((tapgemm2_kernel<256, TG2_EPI_PLAIN>), 232448);
    STAR_SMEM_ATTR((tapgemm2_kernel<128, TG2_EPI_RES>), 232448);
    STAR_SMEM_ATTR((tapgemm2_kernel<160, TG2_EPI_RES>), 232448);
    STAR_SMEM_ATTR((tapgemm2_kernel<128, TG2_EPI_GEGLU>), 232448);
    STAR_SMEM_ATTR((tapgemm2_kernel<256, TG2_EPI_GEGLU>), 232448);
    STAR_SMEM_ATTR(attn_fwd_kernel<false>, AttnSmemT<false>::TOTAL);
    STAR_SMEM_ATTR(attn_fwd_kernel<true>, AttnSmemT<true>::TOTAL);
    STAR_SMEM_ATTR(attn4_fwd_kernel, Attn4Smem::TOTAL);
    STAR_SMEM_ATTR(temporal_attn2_kernel<16>, TA2_WARPS * 3 * 16 * TA2_PITCH);
    STAR_SMEM_ATTR(temporal_attn2_kernel<32>, TA2_WARPS * 3 * 32 * TA2_PITCH);
    STAR_SMEM_ATTR(temporal_attn2_kernel<48>, TA2_WARPS * 3 * 48 * TA2_PITCH);
    STAR_SMEM_ATTR(temporal_attn2_kernel<64>, TA2_WARPS * 3 * 64 * TA2_PITCH);
    STAR_SMEM_ATTR(softmax_rows_kernel, 200 * 1024);
#undef STAR_SMEM_ATTR
    g_sms[device] = prop.multiProcessorCount;
    return 0;
}

int star_init(int device) {
    if (device < 0 || device >= STAR_MAX_DEVICES) return fail("star_init: device index %d out of range", device);
    int prev = -1;
    STAR_CUDA(cudaGetDevice(&prev));
    if (prev != device) STAR_CUDA(cudaSetDevice(device));
    const int rc = star_init_on_current(device);
    if (prev != device && prev >= 0) cudaSetDevice(prev);          // never change the caller's current device
    return rc;
}

int star_linear(const void* A, long long lda, const void* W, const void* bias, const void* rowvec,
                long long rowvec_div, const void* residual, long long ldres, void* out, long long ldo,
                long long rows, int K, int N, int flags, void* stream) {
    return star_linear_ex(A, lda, W, bias, rowvec, rowvec_div, nullptr, residual, ldres, out, ldo, rows, K, N, flags, stream);
}

int star_linear_ex(const void* A, long long lda, const void* W, const void* bias, const void* rowvec,
                   long long rowvec_div, const void* colscale, const void* residual, long long ldres, void* out,
                   long long ldo, long long rows, int K, int N, int flags, void* stream) {
    STAR_CHECK_INIT();
    if (rows <= 0) return 0;
    if (K % 8 || lda % 8) return fail("star_linear: K and lda must be multiples of 8 (K=%d lda=%lld)", K, lda);
    TapDesc d;
    memset(&d, 0, sizeof(d));
    d.A = A;
    d.adim[0] = K; d.adim[1] = rows; d.adim[2] = d.adim[3] = d.adim[4] = 1;
    d.astr[1] = lda; d.astr[2] = d.astr[3] = d.astr[4] = (unsigned long long)lda * rows;
    d.on[0] = (int)rows; d.on[1] = d.on[2] = d.on[3] = 1;
    d.box[0] = TG_BM; d.box[1] = d.box[2] = d.box[3] = 1;
    if (rows > 0x7fffffffll) return fail("star_linear: too many rows");
    d.ntaps = 1;
    d.K = K; d.N = N; d.flags = flags;
    d.W = W; d.bias = bias; d.rowvec = rowvec; d.rowvec_div = rowvec_div; d.residual = residual; d.ldres = ldres;
    d.colscale = colscale;
    d.out = out; d.ldo = ldo;
    return launch_tapgemm(d, (cudaStream_t)stream);
}

int star_conv2d_3x3(const void* X, const void* W9, const void* bias, const void* rowvec, long long rowvec_div, long long ldrowvec,
                    const void* residual, long long ldres, void* out, long long ldo, int BT, int H, int W, int Cin,
                    int Cout, void* stream) {
    STAR_CHECK_INIT();
    if (Cin % 8) return fail("star_conv2d_3x3: Cin must be a multiple of 8");
    TapDesc d;
    memset(&d, 0, sizeof(d));
    d.A = X;
    d.adim[0] = Cin; d.adim[1] = W; d.adim[2] = H; d.adim[3] = BT; d.adim[4] = 1;
    d.astr[1] = Cin; d.astr[2] = (unsigned long long)Cin * W; d.astr[3] = (unsigned long long)Cin * W * H;
    d.astr[4] = (unsigned long long)Cin * W * H * BT;
    d.on[0] = W; d.on[1] = H; d.on[2] = BT; d.on[3] = 1;
    int th = 1, tw = 1;
    best_box_2d(H, W, &th, &tw);
    d.box[0] = tw; d.box[1] = th; d.box[2] = std::max(1, std::min(BT, TG_BM / (tw * th))); d.box[3] = 1;
    d.ntaps = 9;
    for (int r = 0; r < 3; ++r)
        for (int s = 0; s < 3; ++s) {
            d.tap[r * 3 + s][0] = s - 1;
            d.tap[r * 3 + s][1] = r - 1;
        }
    d.K = Cin; d.N = Cout;
    d.W = W9; d.bias = bias; d.rowvec = rowvec; d.rowvec_div = rowvec_div; d.ldrowvec = ldrowvec; d.residual = residual; d.ldres = ldres;
    if (rowvec && ldrowvec % 8) return fail("star_conv2d_3x3: ldrowvec must be a multiple of 8");
    d.out = out; d.ldo = ldo;
    return launch_tapgemm(d, (cudaStream_t)stream);
}

long long star_conv2d_s2p_workspace_bytes(int BT, int H, int W, int Cin, int pad_t, int pad_b, int pad_l, int pad_r) {
    const long long Ho = (H + pad_t + pad_b - 3) / 2 + 1, Wo = (W + pad_l + pad_r - 3) / 2 + 1;
    return (long long)BT * 4 * (Ho + 1) * (Wo + 1) * Cin * 2;
}

long long star_conv2d_s2_workspace_bytes(int BT, int H, int W, int Cin) {
    return star_conv2d_s2p_workspace_bytes(BT, H, W, Cin, 2, 2, 1, 1);
}

int star_conv2d_3x3_s2(const void* X, const void* W9, const void* bias, void* out, long long ldo, void* planes_ws,
                       int BT, int H, int W, int Cin, int Cout, void* stream) {
    return star_conv2d_3x3_s2p(X, W9, bias, out, ldo, planes_ws, BT, H, W, Cin, Cout, 2, 2, 1, 1, stream);
}

int star_conv2d_3x3_s2p(const void* X, const void* W9, const void* bias, void* out, long long ldo, void* planes_ws,
                        int BT, int H, int W, int Cin, int Cout, int pad_t, int pad_b, int pad_l, int pad_r,
                        void* stream) {
    STAR_CHECK_INIT();
    if (Cin % 8) return fail("star_conv2d_3x3_s2p: Cin must be a multiple of 8");
    if (pad_t < 0 || pad_b < 0 || pad_l < 0 || pad_r < 0 || H + pad_t + pad_b < 3 || W + pad_l + pad_r < 3)
        return fail("star_conv2d_3x3_s2p: bad padding");
    const int Ho = (H + pad_t + pad_b - 3) / 2 + 1, Wo = (W + pad_l + pad_r - 3) / 2 + 1, H2 = Ho + 1, W2 = Wo + 1;
    cudaStream_t st = (cudaStream_t)stream;
    const long long n = (long long)BT * 4 * H2 * W2 * (Cin / 8);
    s2_split_kernel<<<grid_for(n, 256), 256, 0, st>>>((const __half*)X, (__half*)planes_ws, BT, H, W, Cin, H2, W2, pad_t, pad_l);
    STAR_LAUNCH_CHECK("s2_split");
    TapDesc d;
    memset(&d, 0, sizeof(d));
    d.A = planes_ws;
    d.adim[0] = Cin; d.adim[1] = W2; d.adim[2] = H2; d.adim[3] = 4; d.adim[4] = BT;
    d.astr[1] = Cin; d.astr[2] = (unsigned long long)Cin * W2; d.astr[3] = (unsigned long long)Cin * W2 * H2;
    d.astr[4] = (unsigned long long)Cin * W2 * H2 * 4;
    d.on[0] = Wo; d.on[1] = Ho; d.on[2] = 1; d.on[3] = BT;
    int th = 1, tw = 1;
    best_box_2d(Ho, Wo, &th, &tw);
    d.box[0] = tw; d.box[1] = th; d.box[2] = 1; d.box[3] = 1;
    d.ntaps = 9;
    for (int r = 0; r < 3; ++r)
        for (int s = 0; s < 3; ++s) {
            d.tap[r * 3 + s][0] = s >> 1;
            d.tap[r * 3 + s][1] = r >> 1;
            d.tap[r * 3 + s][2] = (r & 1) * 2 + (s & 1);
        }
    d.K = Cin; d.N = Cout;
    d.W = W9; d.bias = bias;
    d.out = out; d.ldo = ldo;
    return launch_tapgemm(d, st);
}

int star_conv_t3(const void* X, const void* W3, const void* bias, const void* residual, long long ldres, void* out,
                 long long ldo, int B, int T, long long HW, int Cin, int Cout, void* stream) {
    STAR_CHECK_INIT();
    if (Cin % 8) return fail("star_conv_t3: Cin must be a multiple of 8");
    if (HW > 0x7fffffffll) return fail("star_conv_t3: HW too large");
    TapDesc d;
    memset(&d, 0, sizeof(d));
    d.A = X;
    d.adim[0] = Cin; d.adim[1] = HW; d.adim[2] = T; d.adim[3] = B; d.adim[4] = 1;
    d.astr[1] = Cin; d.astr[2] = (unsigned long long)Cin * HW; d.astr[3] = (unsigned long long)Cin * HW * T;
    d.astr[4] = (unsigned long long)Cin * HW * T * B;
    d.on[0] = (int)HW; d.on[1] = T; d.on[2] = B; d.on[3] = 1;
    d.box[0] = (int)std::min<long long>(TG_BM, HW); d.box[1] = 1; d.box[2] = 1; d.box[3] = 1;
    if (HW < TG_BM) d.box[1] = (int)std::min<long long>(T, TG_BM / HW);     // small latents: several frames per tile
    d.ntaps = 3;
    for (int k = 0; k < 3; ++k) d.tap[k][1] = k - 1;
    d.K = Cin; d.N = Cout;
    d.W = W3; d.bias = bias; d.residual = residual; d.ldres = ldres;
    d.out = out; d.ldo = ldo;
    return launch_tapgemm(d, (cudaStream_t)stream);
}

// Causal Conv3d 3x3x3 of the CogVideoX 3-D VAE (cogvideox-based/sat/vae_modules/cp_enc_dec.py:360-430): X holds T + 2 frames --
// the two frames the reference concatenates in front of the clip (copies of frame 0, or the cache of the previous latent
// chunk, :265-268) followed by the T frames of the clip -- so output frame t reads input frames t, t+1, t+2; the spatial
// zero padding is the TMA out-of-bounds fill.  W27 is [Cout, 3(t), 3(h), 3(w), Cin].
int star_conv3d_causal(const void* X, const void* W27, const void* bias, const void* residual, long long ldres, void* out,
                       long long ldo, int T, int H, int W, int Cin, int Cout, void* stream) {
    STAR_CHECK_INIT();
    if (Cin % 8) return fail("star_conv3d_causal: Cin must be a multiple of 8");
    TapDesc d;
    memset(&d, 0, sizeof(d));
    d.A = X;
    d.adim[0] = Cin; d.adim[1] = W; d.adim[2] = H; d.adim[3] = T + 2; d.adim[4] = 1;
    d.astr[1] = Cin; d.astr[2] = (unsigned long long)Cin * W; d.astr[3] = (unsigned long long)Cin * W * H;
    d.astr[4] = (unsigned long long)Cin * W * H * (T + 2);
    d.on[0] = W; d.on[1] = H; d.on[2] = T; d.on[3] = 1;
    int th = 1, tw = 1;
    best_box_2d(H, W, &th, &tw);
    d.box[0] = tw; d.box[1] = th; d.box[2] = std::max(1, std::min(T, TG_BM / (tw * th))); d.box[3] = 1;
    d.ntaps = 27;
    for (int q = 0; q < 3; ++q)
        for (int r = 0; r < 3; ++r)
            for (int s = 0; s < 3; ++s) {
                int* tp = d.tap[(q * 3 + r) * 3 + s];
                tp[0] = s - 1; tp[1] = r - 1; tp[2] = q;
            }
    d.K = Cin; d.N = Cout;
    d.W = W27; d.bias = bias; d.residual = residual; d.ldres = ldres;
    d.out = out; d.ldo = ldo;
    return launch_tapgemm(d, (cudaStream_t)stream);
}

long long star_conv2d_c4_workspace_bytes(int BT, int H, int W, int Cout) {
    return ((long long)BT * H * W * 64 + (long long)Cout * 64) * 2;
}

int star_conv2d_3x3_c4(const void* X, const void* W9, const void* bias, const void* residual, void* out, void* ws,
                       int BT, int H, int W, int Cout, void* stream) {
    STAR_CHECK_INIT();
    if (Cout % 8) return fail("star_conv2d_3x3_c4: Cout must be a multiple of 8");
    cudaStream_t st = (cudaStream_t)stream;
    const long long rows = (long long)BT * H * W;
    __half* col = (__half*)ws;
    __half* w64 = col + rows * 64;
    pad_w36_kernel<<<(Cout * 64 + 255) / 256, 256, 0, st>>>((const __half*)W9, w64, Cout);
    STAR_LAUNCH_CHECK("pad_w36");
    im2col_c4_kernel<<<grid_for(rows, 256), 256, 0, st>>>((const __half*)X, col, BT, H, W);
    STAR_LAUNCH_CHECK("im2col_c4");
    return star_linear(col, 64, w64, bias, nullptr, 1, residual, Cout, out, Cout, rows, 64, Cout, 0, stream);
}

static int attention_impl(const void* Q, long long ldq, const void* K, long long ldk, const void* V, long long ldv, void* O,
                          long long ldo, int batch, int heads, int Nq, int Nk, int kv_batch_div, float scale, int causal,
                          void* stream) {
    STAR_CHECK_INIT();
    if (ldq % 8 || ldk % 8 || ldv % 8 || ldo % 8) return fail("star_attention: leading dims must be multiples of 8");
    if (Nq <= 0 || Nk <= 0 || batch <= 0) return fail("star_attention: empty problem");
    if (kv_batch_div < 1) kv_batch_div = 1;
    const int kv_batches = (batch + kv_batch_div - 1) / kv_batch_div;
    CUtensorMap tq, tk, tv;
    unsigned box[3] = {AT_D, AT_BQ, 1};
    {
        unsigned long long dims[3] = {(unsigned long long)heads * AT_D, (unsigned long long)Nq, (unsigned long long)batch};
        unsigned long long str[3] = {1, (unsigned long long)ldq, (unsigned long long)ldq * Nq};
        if (make_tmap(&tq, Q, 3, dims, str, box)) return 1;
    }
    {
        unsigned long long dims[3] = {(unsigned long long)heads * AT_D, (unsigned long long)Nk, (unsigned long long)kv_batches};
        unsigned long long strk[3] = {1, (unsigned long long)ldk, (unsigned long long)ldk * Nk};
        unsigned long long strv[3] = {1, (unsigned long long)ldv, (unsigned long long)ldv * Nk};
        if (make_tmap(&tk, K, 3, dims, strk, box)) return 1;
        if (make_tmap(&tv, V, 3, dims, strv, box)) return 1;
    }
    AttnParams p;
    p.Nq = Nq; p.Nk = Nk; p.kv_batch_div = kv_batch_div; p.causal = causal;
    p.scale_log2 = scale * 1.4426950408889634f;
    p.out = (__half*)O; p.ldo = ldo;
    if (heads > 65535 || batch > 65535) return fail("star_attention: grid too large");
    cudaStream_t st = (cudaStream_t)stream;
    // Multi-tile problems (spatial self-attention): two 128-row query tiles per CTA, row-split softmax, every exponential on
    // the MUFU (in-step A/B on the full model: profiles/r01_bench_ab_attention.log).  Single-KV-tile problems (text
    // cross-attention, tiny latents): the one-tile kernel, two CTAs per SM.
    if (Nk > AT_BKV && Nq > AT_BQ && !causal) {
        dim3 grid((Nq + 255) / 256, heads, batch);
        attn4_fwd_kernel<<<grid, A4S_THREADS, Attn4Smem::TOTAL, st>>>(tq, tk, tv, p);
        STAR_LAUNCH_CHECK("attn4_fwd");
        return 0;
    }
    dim3 grid((Nq + AT_BQ - 1) / AT_BQ, heads, batch);
    if (Nk <= AT_BKV) attn_fwd_kernel<true><<<grid, AT_THREADS, AttnSmemT<true>::TOTAL, st>>>(tq, tk, tv, p);
    else attn_fwd_kernel<false><<<grid, AT_THREADS, AttnSmemT<false>::TOTAL, st>>>(tq, tk, tv, p);
    STAR_LAUNCH_CHECK("attn_fwd");
    return 0;
}

int star_attention(const void* Q, long long ldq, const void* K, long long ldk, const void* V, long long ldv, void* O,
                   long long ldo, int batch, int heads, int Nq, int Nk, int kv_batch_div, float scale, void* stream) {
    return attention_impl(Q, ldq, K, ldk, V, ldv, O, ldo, batch, heads, Nq, Nk, kv_batch_div, scale, 0, stream);
}

// causal self-attention (query i attends keys 0..i): the text tower's attn_mask (embedder.py:57, open_clip build_attention_mask)
int star_attention_causal(const void* Q, long long ldq, const void* K, long long ldk, const void* V, long long ldv, void* O,
                          long long ldo, int batch, int heads, int N, float scale, void* stream) {
    return attention_impl(Q, ldq, K, ldk, V, ldv, O, ldo, batch, heads, N, N, 1, scale, 1, stream);
}

int star_temporal_attention(const void* QKV, long long ld, void* O, long long ldo, int B, int T, long long HW,
                            int heads, int Ci, float scale, void* stream) {
    STAR_CHECK_INIT();
    if (T > TA2_MAXT || T < 1) return fail("star_temporal_attention: T=%d outside [1, %d]", T, TA2_MAXT);
    if (ld % 8 || ldo % 8 || Ci % 8) return fail("star_temporal_attention: ld/ldo/Ci must be multiples of 8");
    if ((reinterpret_cast<uintptr_t>(QKV) | reinterpret_cast<uintptr_t>(O)) % 16) return fail("star_temporal_attention: pointers must be 16-byte aligned");
    const long long items = (long long)B * HW * heads;
    cudaStream_t st = (cudaStream_t)stream;
    const int tp = (T + 15) / 16 * 16;
    const unsigned grid = (unsigned)std::min<long long>((items + TA2_WARPS - 1) / TA2_WARPS, (long long)num_sms() * 2);
    const size_t smem = (size_t)TA2_WARPS * 3 * tp * TA2_PITCH;
#define STAR_TA2(TPV) temporal_attn2_kernel<TPV><<<grid, TA2_WARPS * 32, smem, st>>>((const __half*)QKV, ld, (__half*)O, ldo, B, T, HW, heads, Ci, scale)
    switch (tp) {
        case 16: STAR_TA2(16); break;
        case 32: STAR_TA2(32); break;
        case 48: STAR_TA2(48); break;
        default: STAR_TA2(64); break;
    }
#undef STAR_TA2
    STAR_LAUNCH_CHECK("temporal_attn2");
    return 0;
}

long long star_groupnorm_workspace_bytes(int nsamples, int C) {
    return (long long)nsamples * 32 * 2 * 8 + (long long)nsamples * C * 2 * 4;
}

int star_groupnorm(const void* X, const void* gamma, const void* beta, void* out, int nsamples,
                   long long rows_per_sample, int C, float eps, int silu, void* workspace, void* stream) {
    if (C % 256 && C % 32) return fail("star_groupnorm: C must be a multiple of 32");
    if (C % 8) return fail("star_groupnorm: C must be a multiple of 8");
    if (C / 8 > GN_THREADS) return fail("star_groupnorm: C too large");
    cudaStream_t st = (cudaStream_t)stream;
    double* stats = (double*)workspace;
    float* ab = (float*)((char*)workspace + (size_t)nsamples * 32 * 2 * 8);
    STAR_CUDA(cudaMemsetAsync(stats, 0, (size_t)nsamples * 32 * 2 * 8, st));
    const long long total_rows = rows_per_sample * nsamples;
    if (C / 8 <= GN2_THREADS) {
        // persistent CTAs over contiguous slab ranges: statistics / (a, b) stay in registers across slabs
        Gn2Range rg;
        rg.slabs_per_sample = (rows_per_sample + GN2_SLAB - 1) / GN2_SLAB;
        rg.total_slabs = rg.slabs_per_sample * nsamples;
        const int lanes2 = GN2_THREADS / (C / 8);
        const size_t smem2 = (size_t)lanes2 * C * 2 * sizeof(float);
        const unsigned grid2 = (unsigned)std::min<long long>(rg.total_slabs, (long long)num_sms() * 8);
        gn_stats2_kernel<<<grid2, GN2_THREADS, smem2, st>>>((const __half*)X, stats, rows_per_sample, C, rg);
        STAR_LAUNCH_CHECK("gn_stats2");
        gn_finalize_kernel<<<nsamples, 256, 0, st>>>(stats, (const __half*)gamma, (const __half*)beta, ab, rows_per_sample, C, eps);
        STAR_LAUNCH_CHECK("gn_finalize");
        gn_apply2_kernel<<<grid2, GN2_THREADS, 0, st>>>((const __half*)X, ab, (__half*)out, rows_per_sample, C, silu, rg);
        STAR_LAUNCH_CHECK("gn_apply2");
        return 0;
    }
    const int lanes = std::max(1, GN_THREADS / (C / 8));
    const size_t smem = (size_t)lanes * C * 2 * sizeof(float);
    dim3 grid((unsigned)((rows_per_sample + GN_SLAB - 1) / GN_SLAB), nsamples);
    gn_stats_kernel<<<grid, GN_THREADS, smem, st>>>((const __half*)X, stats, rows_per_sample, C);
    STAR_LAUNCH_CHECK("gn_stats");
    gn_finalize_kernel<<<nsamples, 256, 0, st>>>(stats, (const __half*)gamma, (const __half*)beta, ab, rows_per_sample, C, eps);
    STAR_LAUNCH_CHECK("gn_finalize");
    gn_apply_kernel<<<grid_for(total_rows * (C / 8), 256), 256, 0, st>>>((const __half*)X, ab, (__half*)out, rows_per_sample,
                                                                          total_rows, C, silu);
    STAR_LAUNCH_CHECK("gn_apply");
    return 0;
}

// SpatialNorm3D of the CogVideoX 3-D VAE decoder (cp_enc_dec.py:451-510): out = GroupNorm32(X) * Ymod[src] + Bmod[src] (+ SiLU)
// over ONE clip of T x H x W rows; Ymod / Bmod = conv_y(zq) / conv_b(zq) at latent resolution (Tl, Hl, Wl) (see
// gn_apply_mod_kernel), row pitch ldmod.  Workspace: star_groupnorm_workspace_bytes(1, C).
int star_groupnorm_mod(const void* X, const void* gamma, const void* beta, const void* Ymod, const void* Bmod, long long ldmod,
                       void* out, int T, int H, int W, int Tl, int Hl, int Wl, int C, float eps, int silu, void* workspace, void* stream) {
    if (C % 32) return fail("star_groupnorm_mod: C must be a multiple of 32");
    if (C / 8 > GN2_THREADS) return fail("star_groupnorm_mod: C too large");
    if (H % Hl || W % Wl) return fail("star_groupnorm_mod: feature size must be a multiple of the latent size");
    if (ldmod % 8 || ldmod < C) return fail("star_groupnorm_mod: ldmod must be a multiple of 8 and >= C");
    const bool split = T > 1 && (T & 1);
    if (split ? ((T - 1) % std::max(1, Tl - 1) != 0 || Tl < 2) : (T % Tl != 0))
        return fail("star_groupnorm_mod: T=%d is not an integer multiple of the latent T=%d", T, Tl);
    cudaStream_t st = (cudaStream_t)stream;
    double* stats = (double*)workspace;
    float* ab = (float*)((char*)workspace + (size_t)32 * 2 * 8);
    STAR_CUDA(cudaMemsetAsync(stats, 0, (size_t)32 * 2 * 8, st));
    const long long rows = (long long)T * H * W;
    Gn2Range rg;
    rg.slabs_per_sample = (rows + GN2_SLAB - 1) / GN2_SLAB;
    rg.total_slabs = rg.slabs_per_sample;
    const int lanes2 = GN2_THREADS / (C / 8);
    const size_t smem2 = (size_t)lanes2 * C * 2 * sizeof(float);
    const unsigned grid2 = (unsigned)std::min<long long>(rg.total_slabs, (long long)num_sms() * 8);
    gn_stats2_kernel<<<grid2, GN2_THREADS, smem2, st>>>((const __half*)X, stats, rows, C, rg);
    STAR_LAUNCH_CHECK("gn_stats2");
    gn_finalize_kernel<<<1, 256, 0, st>>>(stats, (const __half*)gamma, (const __half*)beta, ab, rows, C, eps);
    STAR_LAUNCH_CHECK("gn_finalize");
    if (rows > 0x7fffffffll) return fail("star_groupnorm_mod: more than 2^31 rows");
    auto log2_exact = [](int q) { int s = 0; while ((1 << s) < q) ++s; return (1 << s) == q ? s : -1; };
    GnModGeom gm{T, H, W, Tl, Hl, Wl, split ? 1 : 0, log2_exact(H / Hl), log2_exact(W / Wl)};
    gn_apply_mod_kernel<<<grid2, GN2_THREADS, 0, st>>>((const __half*)X, ab, (const __half*)Ymod, (const __half*)Bmod,
                                                       ldmod, (__half*)out, rows, C, silu, rg, gm);
    STAR_LAUNCH_CHECK("gn_apply_mod");
    return 0;
}

int star_layernorm(const void* X, const void* gamma, const void* beta, void* out, long long rows, int C, float eps,
                   int gate_mode, const void* gate, float w0, float w1, void* stream) {
    if (C % 8 || C / 8 > 32 * 12) return fail("star_layernorm: unsupported C=%d", C);
    if (C == 320 || C == 640) {
        const int rpw = C == 320 ? 4 : 2;
        const long long groups = (rows + rpw - 1) / rpw;
        const unsigned g2 = (unsigned)std::min<long long>((groups + 7) / 8, (long long)num_sms() * 6);
        if (C == 320)
            layernorm_sub_kernel<8><<<g2, 256, 0, (cudaStream_t)stream>>>((const __half*)X, (const __half*)gamma, (const __half*)beta,
                                                                          (__half*)out, rows, eps, gate_mode, (const __half*)gate, w0, w1);
        else
            layernorm_sub_kernel<16><<<g2, 256, 0, (cudaStream_t)stream>>>((const __half*)X, (const __half*)gamma, (const __half*)beta,
                                                                           (__half*)out, rows, eps, gate_mode, (const __half*)gate, w0, w1);
        STAR_LAUNCH_CHECK("layernorm_sub");
        return 0;
    }
    const int wpb = 8;
    const long long want = (rows + wpb - 1) / wpb;
    const unsigned grid = (unsigned)std::min<long long>(want, (long long)num_sms() * 6);
    const int oct = (C / 8 + 31) / 32;
#define STAR_LN_LAUNCH(N)                                                                                          \
    layernorm_kernel<N><<<grid, wpb * 32, 0, (cudaStream_t)stream>>>((const __half*)X, (const __half*)gamma,          \
                                                                     (const __half*)beta, (__half*)out, rows, C, eps, \
                                                                     gate_mode, (const __half*)gate, w0, w1)
    if (oct <= 2) STAR_LN_LAUNCH(2);
    else if (oct <= 3) STAR_LN_LAUNCH(3);
    else if (oct <= 5) STAR_LN_LAUNCH(5);
    else STAR_LN_LAUNCH(12);
#undef STAR_LN_LAUNCH
    STAR_LAUNCH_CHECK("layernorm");
    return 0;
}

int star_liem_spatial_gate(const void* X, const void* w98, void* mm_ws, void* gate, int BT, int H, int W, int C,
                           void* stream) {
    if (C % 8) return fail("star_liem_spatial_gate: C must be a multiple of 8");
    cudaStream_t st = (cudaStream_t)stream;
    const long long rows = (long long)BT * H * W;
    liem_reduce_kernel<<<(unsigned)std::min<long long>((rows + 7) / 8, (long long)num_sms() * 8), 256, 0, st>>>((const __half*)X, (__half*)mm_ws, rows, C);
    STAR_LAUNCH_CHECK("liem_reduce");
    liem_conv7_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, st>>>((const __half*)mm_ws, (const __half*)w98, (__half*)gate,
                                                                       BT, H, W);
    STAR_LAUNCH_CHECK("liem_conv7");
    return 0;
}

int star_row_gate(const void* X, void* out, long long rows, int C, int mode, const void* gate, float w0, float w1,
                  void* stream) {
    if (C % 8) return fail("star_row_gate: C must be a multiple of 8");
    if (mode != 1 && mode != 2) return fail("star_row_gate: mode must be 1 (external gate) or 2 (temporal LIEM)");
    const unsigned grid = (unsigned)std::min<long long>((rows + 7) / 8, (long long)num_sms() * 8);
    row_gate_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const __half*)X, (__half*)out, rows, C, mode, (const __half*)gate, w0, w1);
    STAR_LAUNCH_CHECK("row_gate");
    return 0;
}

int star_qk_ln_rope(void* QKV, long long ld, long long rows, int heads, int koff, const void* qg, const void* qb,
                    const void* kg, const void* kb, const void* cos_f32, const void* sin_f32, int seq, int text_len,
                    float eps, void* stream) {
    if (ld % 8 || koff % 8) return fail("star_qk_ln_rope: ld and koff must be multiples of 8");
    const long long threads = rows * heads * 2 * 8;
    qk_ln_rope_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        (__half*)QKV, ld, rows, heads, koff, (const __half*)qg, (const __half*)qb, (const __half*)kg, (const __half*)kb,
        (const float*)cos_f32, (const float*)sin_f32, seq, text_len, eps);
    STAR_LAUNCH_CHECK("qk_ln_rope");
    return 0;
}

int star_concat_add(const void* a, int Ca, const void* b, const void* c, int Cb, void* out, long long rows,
                    void* stream) {
    if (Ca % 8 || Cb % 8) return fail("star_concat_add: channel counts must be multiples of 8");
    const long long n = rows * ((Ca + Cb) / 8);
    concat_add_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>((const __half*)a, Ca, (const __half*)b,
                                                                           (const __half*)c, Cb, (__half*)out, rows);
    STAR_LAUNCH_CHECK("concat_add");
    return 0;
}

int star_add(const void* a, const void* b, void* out, long long n, void* stream) {
    if (n % 8) return fail("star_add: n must be a multiple of 8");
    add_kernel<<<grid_for(n / 8, 256), 256, 0, (cudaStream_t)stream>>>((const __half*)a, (const __half*)b, (__half*)out, n / 8);
    STAR_LAUNCH_CHECK("add");
    return 0;
}

int star_time_avgpool2(const void* X, void* out, int T, long long HW, int C, void* stream) {
    if (C % 8) return fail("star_time_avgpool2: C must be a multiple of 8");
    if (T < 2) return fail("star_time_avgpool2: needs at least two frames");
    const long long per8 = HW * C / 8;
    const int To = (T & 1) ? (T + 1) / 2 : T / 2;
    time_avgpool2_kernel<<<grid_for(per8 * To, 256), 256, 0, (cudaStream_t)stream>>>((const __half*)X, (__half*)out, T, per8);
    STAR_LAUNCH_CHECK("time_avgpool2");
    return 0;
}

int star_upsample2x(const void* X, void* out, int BT, int H, int W, int C, int crop_rows, void* stream) {
    if (C % 8) return fail("star_upsample2x: C must be a multiple of 8");
    if (crop_rows != 0 && crop_rows != 1) return fail("star_upsample2x: crop_rows must be 0 or 1");
    const long long n = (long long)BT * (2 * H - 2 * crop_rows) * (2 * W) * (C / 8);
    upsample2x_crop_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>((const __half*)X, (__half*)out, BT, H, W, C, crop_rows);
    STAR_LAUNCH_CHECK("upsample2x");
    return 0;
}

int star_upsample2x_crop(const void* X, void* out, int BT, int H, int W, int C, void* stream) {
    return star_upsample2x(X, out, BT, H, W, C, 1, stream);
}

int star_softmax_rows(void* S, long long ld, long long rows, int cols, void* stream) {
    STAR_CHECK_INIT();
    if (rows <= 0) return 0;
    if (ld % 8 || reinterpret_cast<uintptr_t>(S) % 16) return fail("star_softmax_rows: rows must be 16-byte aligned (ld %% 8 == 0)");
    if (cols <= 0 || cols > ld) return fail("star_softmax_rows: need 0 < cols <= ld");
    const size_t smem = ((size_t)cols * 2 + 15) / 16 * 16;
    if (smem > 200 * 1024) return fail("star_softmax_rows: %d columns do not fit in shared memory", cols);
    if (rows > 0x7fffffffll) return fail("star_softmax_rows: too many rows");
    softmax_rows_kernel<<<(unsigned)rows, 256, smem, (cudaStream_t)stream>>>((__half*)S, ld, cols);
    STAR_LAUNCH_CHECK("softmax_rows");
    return 0;
}

int star_vae_head(const void* X, long long ldx, const void* W27, const void* bias3, void* out, int B, int T,
                  long long HW, void* stream) {
    if (ldx < 3) return fail("star_vae_head: ldx must be >= 3");
    const long long n = (long long)B * T * HW;
    vae_head_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>((const __half*)X, ldx, (const __half*)W27,
                                                                        (const __half*)bias3, (__half*)out, B, T, HW);
    STAR_LAUNCH_CHECK("vae_head");
    return 0;
}

int star_nchw5_to_tokens(const void* x_f32, void* out, int B, int C, int F, long long HW, void* stream) {
    const long long n = (long long)B * F * HW;
    nchw5_to_tokens_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>((const float*)x_f32, (__half*)out, B, C, F, HW);
    STAR_LAUNCH_CHECK("nchw5_to_tokens");
    return 0;
}

int star_tokens_to_nchw5(const void* x, long long ldx, void* out, int B, int C, int F, long long HW, void* stream) {
    const long long n = (long long)B * F * HW;
    tokens_to_nchw5_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>((const __half*)x, ldx, (__half*)out, B, C, F, HW);
    STAR_LAUNCH_CHECK("tokens_to_nchw5");
    return 0;
}

int star_bilinear_pad(const void* x_f32, void* out_f32, long long NC, int h, int w, int H, int W, int pad_l, int pad_r,
                      int pad_t, int pad_b, float pad_value, void* stream) {
    if (NC <= 0 || h <= 0 || w <= 0 || H <= 0 || W <= 0 || pad_l < 0 || pad_r < 0 || pad_t < 0 || pad_b < 0)
        return fail("star_bilinear_pad: bad geometry");
    const int Hp = H + pad_t + pad_b, Wp = W + pad_l + pad_r;
    const long long n = NC * Hp * Wp;
    bilinear_pad_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>((const float*)x_f32, (float*)out_f32, NC, h, w, H, W,
                                                                            pad_l, pad_t, Hp, Wp, (float)h / (float)H,
                                                                            (float)w / (float)W, pad_value);
    STAR_LAUNCH_CHECK("bilinear_pad");
    return 0;
}

long long star_adain_workspace_bytes(int C, int F) { return (long long)C * F * 2 * 2 * 8; }

int star_adain_color_fix(const void* video_f32, const void* source_f32, void* out_f32, void* out_u8, int C, int F, long long HW,
                         long long src_hw, void* workspace, void* stream) {
    if (C < 1 || C > 4 || F < 1 || HW < 2 || src_hw < 2) return fail("star_adain_color_fix: bad geometry (C <= 4)");
    if ((out_f32 == nullptr) == (out_u8 == nullptr)) return fail("star_adain_color_fix: pass exactly one of out_f32 / out_u8");
    if (F > 65535) return fail("star_adain_color_fix: too many frames");
    cudaStream_t st = (cudaStream_t)stream;
    double* tgt = (double*)workspace;
    double* src = tgt + (size_t)C * F * 2;
    STAR_CUDA(cudaMemsetAsync(workspace, 0, (size_t)star_adain_workspace_bytes(C, F), st));
    const unsigned gt = (unsigned)std::min<long long>((HW + 255) / 256, 256), gs = (unsigned)std::min<long long>((src_hw + 255) / 256, 256);
    plane_stats_kernel<<<dim3(gt, C * F), 256, 0, st>>>((const float*)video_f32, HW, 1, tgt);
    STAR_LAUNCH_CHECK("plane_stats(target)");
    plane_stats_kernel<<<dim3(gs, C * F), 256, 0, st>>>((const float*)source_f32, src_hw, 0, src);
    STAR_LAUNCH_CHECK("plane_stats(source)");
    adain_apply_kernel<<<dim3((unsigned)std::min<long long>((HW + 255) / 256, 1024), F), 256, 0, st>>>(
        (const float*)video_f32, (float*)out_f32, (unsigned char*)out_u8, C, F, HW, src_hw, tgt, src);
    STAR_LAUNCH_CHECK("adain_apply");
    return 0;
}

long long star_cfg_x0_workspace_bytes(int samples) { return (long long)samples * 4 * 8; }

int star_cfg_x0(const void* y_out, const void* u_out, const void* xt_f32, void* x0_f32, void* guided_out,
                float guide_scale, float guide_rescale, const void* alpha_f32, const void* sigma_f32, int samples,
                long long per_sample, void* workspace, void* stream) {
    if (samples <= 0 || per_sample <= 1) return fail("star_cfg_x0: empty problem");
    if (samples > 65535) return fail("star_cfg_x0: too many samples");
    cudaStream_t st = (cudaStream_t)stream;
    const int has_rescale = guide_rescale >= 0.f;
    double* stats = (double*)workspace;
    const unsigned gx = (unsigned)std::min<long long>((per_sample + 255) / 256, (long long)num_sms() * 8);
    if (has_rescale) {
        if (!workspace) return fail("star_cfg_x0: the std-ratio rescale needs a workspace");
        STAR_CUDA(cudaMemsetAsync(stats, 0, (size_t)samples * 4 * 8, st));
        cfg_stats_kernel<<<dim3(gx, samples), 256, 0, st>>>((const __half*)y_out, (const __half*)u_out, guide_scale, per_sample, stats);
        STAR_LAUNCH_CHECK("cfg_stats");
    }
    cfg_x0_kernel<<<dim3(gx, samples), 256, 0, st>>>((const __half*)y_out, (const __half*)u_out, (const float*)xt_f32,
                                                     (float*)x0_f32, (__half*)guided_out, guide_scale, guide_rescale,
                                                     has_rescale, (const float*)alpha_f32, (const float*)sigma_f32, per_sample, stats);
    STAR_LAUNCH_CHECK("cfg_x0");
    return 0;
}

#if STAR_GEMM_TRACE
// experiment builds only (tools/gemm_trace.py): copy CTA 0's role timelines to the host and reset them
int star_debug_read_trace(long long* host_dst, int* host_counts) {
    STAR_CUDA(cudaDeviceSynchronize());
    STAR_CUDA(cudaMemcpyFromSymbol(host_dst, g_tg2_trace, sizeof(long long) * 3 * 4096));
    STAR_CUDA(cudaMemcpyFromSymbol(host_counts, g_tg2_trace_n, sizeof(int) * 3));
    int zero[3] = {0, 0, 0};
    STAR_CUDA(cudaMemcpyToSymbol(g_tg2_trace_n, zero, sizeof(zero)));
    return 0;
}
#endif

#if STAR_ATTN_TRACE
// experiment builds only (tools/attn_trace.py): softmax-phase timelines of CTA (0,0,0) of the spatial-attention kernel
int star_debug_read_attn_trace(long long* host_dst, int* host_counts) {
    STAR_CUDA(cudaDeviceSynchronize());
    STAR_CUDA(cudaMemcpyFromSymbol(host_dst, g_a4_trace, sizeof(long long) * 2 * 8192));
    STAR_CUDA(cudaMemcpyFromSymbol(host_counts, g_a4_trace_n, sizeof(int) * 2));
    int zero[2] = {0, 0};
    STAR_CUDA(cudaMemcpyToSymbol(g_a4_trace_n, zero, sizeof(zero)));
    return 0;
}
#endif

int star_sinusoidal(const void* t_i64, void* out, int B, int dim, void* stream) {
    const int n = B * (dim / 2);
    sinusoidal_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>((const long long*)t_i64, (__half*)out, B, dim);
    STAR_LAUNCH_CHECK("sinusoidal");
    return 0;
}

int star_silu(const void* x, void* out, long long n, void* stream) {
    silu_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>((const __half*)x, (__half*)out, n);
    STAR_LAUNCH_CHECK("silu");
    return 0;
}

}  // extern "C"
