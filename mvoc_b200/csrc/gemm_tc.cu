// Dense work of the UNet on tcgen05 tensor cores (SURVEY §8 f1): 3x3 convolutions, temporal (3,1,1) convolutions
// and every Linear / 1x1 conv as ONE persistent, warp-specialised implicit-GEMM kernel on channels-last bf16 / fp16
// activations.  Replaces what the reference leaves to cuDNN / cuBLAS:
//   resnet conv1 / conv2 (+ 1x1 shortcut, + residual)      i2vgen-xl/pnp_utils.py:939, :968, :1011-1018
//   TemporalConvLayer conv1..4 (+ identity)                 i2vgen-xl/pnp_utils.py:1048-1053
//   to_q / to_k / to_v / to_out, proj_in / proj_out         i2vgen-xl/pnp_utils.py:604-612, :692, :191, :206, :432, :503
//   GEGLU feed-forward                                      i2vgen-xl/pnp_utils.py:335
//   CLIP image tower mlp.fc1 + GELU (Linear with the exact GELU in the epilogue; mvoc_b200/clip.py)
//
// Formulation.  out[row, n] = sum_{src, tap, k} A_src[row + shift(tap), k] * W_src[tap, n, k]  (+ bias[n]) (+ residual)
// where the rows of A are the pixels of a channels-last activation viewed as a 4-D tensor [K, d1, d2, d3]:
//   conv3x3     : [Cin, W, H, N], 9 taps shifting (d1, d2) by (-1..1, -1..1)
//   temporal    : [Cin, S, T, B], 3 taps shifting d2 (the frame) by -1..1
//   linear      : [K, M, 1, 1],   1 tap
//   conv3x3 s2  : [Cout rows on the OUTPUT grid Wo, Ho, N]; the A map reads the input [Cin, W, H, N] with TMA
//                 traversal stride 2 along (d1, d2), so a box {64, 2 b1, 2 b2, b3} delivers the b1 x b2 x b3 = 128
//                 input pixels under the tile's output pixels, and tap (kh, kw) starts at (2 ox0 + kw - pad,
//                 2 oy0 + kh - pad).  Tiles, MMAs and the epilogue are those of the stride-1 conv.
// A tile of 128 rows is a TMA box {64 channels, b1, b2, b3} whose start coordinate is moved by the tap shift;
// rows that fall outside the tensor are ZERO-FILLED by TMA, which IS the convolution's padding — no im2col
// buffer, no halo copy.  A second (A, W) source appended to the K loop fuses the resnet's 1x1 shortcut conv
// into conv2's accumulator.
//
// CTA (320 threads, one per SM, persistent over tiles, static round-robin schedule):
//   warp 0     TMA producer: ring of kStages {A 128x64, W BNx64} 128-byte-swizzled stages
//   warp 1     MMA issuer (one lane): tcgen05.mma 128 x BN x 16 into one of TWO accumulator buffers in TMEM,
//              so the epilogue of tile i overlaps the main loop of tile i+1; owns the TMEM allocation
//   warps 2-9  epilogue, two warps per TMEM lane quarter taking alternate 32-column slabs: thread = TMEM lane =
//              output row; tcgen05.ld -> + bias -> (+ residual, TMA-loaded into the staging buffer two slabs ahead)
//              -> (GEGLU) -> bf16 -> swizzled smem -> TMA store of the warp's 32-row box
// kTwoCta: the same kernel as a CTA PAIR (cluster of 2, tcgen05 cta_group::2): one 256 x BN tile per pair, each
// CTA stages its own 128 rows of A and HALF of the weight tile, the leader issues M = 256 MMAs that read both
// halves — weight traffic from L2 per CTA halves.
#include <cuda.h>
#include <type_traits>
#include "common.cuh"
#include "ptx.cuh"

namespace mvoc {
namespace gemm {

// Relative cost of one 64-element K chunk of a tile by tile width, measured on B200 with ONE convolution whose Cout
// every width divides (profiles/r02_gemm_width_*.txt: time per tile-chunk = width / TFLOP/s).  The striking fact:
// it is nearly independent of the width — a tcgen05.mma with both operands in shared memory takes ~128 clocks per
// 128-row K = 16 step whatever N <= 256 is (the A-operand read paces it), so a tile's efficiency is N / 256 and the
// number of column tiles is what matters.  256-wide single-CTA tiles pay extra for the shared-memory fill.
static double chunk_cost(int w, bool pair) {
    switch (w) {
        case 256: return pair ? 152.0 : 191.0;
        case 192: return pair ? 133.0 : 146.0;
        case 160: return pair ? 143.0 : 146.0;
        case 128: return pair ? 136.0 : 138.0;
        default: return pair ? 119.0 : 121.0;   // 64
    }
}

constexpr int BM = 128;                    // rows (pixels) per CTA tile
constexpr int KC = 64;                     // K elements per stage = one 128-byte swizzled row
constexpr int A_BYTES = BM * KC * 2;       // 16 KB
constexpr int SMEM_LIMIT = 232448;         // 227 KB per CTA
constexpr uint32_t TMEM_COLS = 512;
constexpr int MAX_TAPS = 9;

enum Epilogue { EPI_LINEAR = 0, EPI_GEGLU = 1, EPI_GELU = 2 };   // GELU: the Linear's tile, then gelu(out)

template <int BN_, bool kTwoCta_, int kEpi_>
struct Cfg {
    static constexpr int BN = BN_;
    static constexpr bool kTwoCta = kTwoCta_;
    static constexpr int kEpi = kEpi_;
    static constexpr int B_ROWS = kTwoCta ? BN / 2 : BN;     // weight rows THIS CTA stages
    static constexpr int B_BYTES = B_ROWS * KC * 2;
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int OUT_COLS = kEpi == EPI_GEGLU ? BN / 2 : BN;   // output columns of a tile
    // Epilogue: 32-column slabs (64-byte staging rows, 64B swizzle) on EIGHT warps, two per TMEM lane quarter taking
    // alternate slabs.  With four warps each one sat alone on its scheduler and issued one instruction per ~6.6
    // clocks (ncu, profiles/r02_ncu_linear_summary.txt): a 192-column tile cost ~7000 clocks of epilogue against
    // 2560 clocks of MMAs at K = 320, which is what bounded every short-K Linear.
    static constexpr int SLAB = 32;
    static constexpr int SLABS = OUT_COLS / SLAB;
    static constexpr int WSLAB_BYTES = 32 * SLAB * 2;        // one warp's 32 rows of one slab: 2 KB
    static constexpr int EPI_WARPS = 8;
    static constexpr int HALVES = EPI_WARPS / 4;
    static constexpr int THREADS = 64 + 32 * EPI_WARPS;
    // Staging buffers per epilogue warp = RES_AHEAD + ST_PENDING: while slab g is processed the residual of slab
    // g + RES_AHEAD is being TMA-loaded and up to ST_PENDING TMA stores may still be reading their buffers (lanes
    // other than lane 0 run one slab ahead of its wait, hence ST_PENDING <= N_OUT - 2).  Deeper variants (3 ahead,
    // 3 pending) were measured and only cost pipeline stages (profiles/r02_gemm_epilogue_experiments.txt).
    static constexpr int RES_AHEAD = 2;
    static constexpr int ST_PENDING = 1;
    static constexpr int N_OUT = RES_AHEAD + ST_PENDING;
    static constexpr int out_off = 0;                        // staging first: 1024-byte aligned like the stages
    static constexpr int stage_off = EPI_WARPS * N_OUT * WSLAB_BYTES;
    static constexpr int kStagesFit = (SMEM_LIMIT - stage_off - 512) / STAGE_BYTES;
    static constexpr int kStages = kStagesFit > 8 ? 8 : kStagesFit;
    static constexpr int bar_off = stage_off + kStages * STAGE_BYTES;
    // barriers: full[kStages], empty[kStages], acc_full[2], acc_empty[2], res_full[EPI_WARPS][N_OUT]
    static constexpr int n_bars = 2 * kStages + 4 + EPI_WARPS * N_OUT;
    static constexpr int tmem_ptr_off = bar_off + n_bars * 8;
    static constexpr int alloc = tmem_ptr_off + 16;
    static_assert(BN % 32 == 0 && BN >= 64 && BN <= 256, "BN: multiple of 32 in [64, 256]");
    static_assert(OUT_COLS % SLAB == 0, "tile columns must be whole slabs");
    static_assert(B_BYTES % 1024 == 0, "weight stage must keep the 1024-byte swizzle-atom alignment");
    static_assert(kStages >= 3, "too few pipeline stages");
    static_assert(alloc <= SMEM_LIMIT, "shared memory budget exceeded");
    static_assert(2 * BN <= (int)TMEM_COLS, "two accumulator buffers must fit in TMEM");
};

struct Params {
    int total_tiles;           // tiles (1-CTA) or tile PAIRS (2-CTA) of the whole problem
    int n_tiles;               // column tiles
    int t1, t2;                // row tiles along d1 and d2 (d3 follows)
    int b1, b2, b3;            // row box, b1 * b2 * b3 == 128
    int n_src;                 // 1 or 2 (A, W) sources in the K loop
    int k_chunks[2];           // K / 64 per source
    int taps[2];
    int8_t off[2][MAX_TAPS][3];   // coordinate shift of (d1, d2, d3) per tap
    int tail_cols;             // > 0: the LAST column tile is only this wide (multiple of 64; N % BN); its MMAs run at
                               // N = tail_cols and the epilogue skips the slabs beyond it
    int gate_off;              // GEGLU: row of W where the gate half starts (F)
    int has_res;
    int a_stride;              // A coordinate of a tile row = a_stride x its output coordinate (d1, d2) + tap shift
    int dbg;                   // timing experiments only (results are garbage): 1 = never reload the weight stage,
                               // 2 = never reload the activation stage, 4 = no TMA stores, 8 = no epilogue work at
                               // all (accumulators released at once)  (variant bits 20..23)
    const void* bias;          // [N] (GEGLU: [2F]) in the activation dtype, or nullptr
};

// ---- PTX pieces this kernel adds to ptx.cuh --------------------------------------------------------------------
constexpr uint32_t PEER_MASK = 0xFEFFFFFFu;   // clears the CTA-rank bit of a shared::cluster address in a CTA pair

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
template <bool kTwoCta>
__device__ __forceinline__ void tma_load_tile(uint32_t dst, const void* tmap, uint32_t bar, int c0, int c1, int c2,
                                              int c3) {
    if (kTwoCta) {
        // executed by both CTAs of the pair; the transaction bytes land on the LEADER's barrier
        asm volatile(
            "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes "
            "[%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(dst),
            "l"(tmap), "r"(bar & PEER_MASK), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
            : "memory");
    } else {
        ptx::tma_load_4d(dst, tmap, bar, c0, c1, c2, c3);
    }
}
__device__ __forceinline__ void tma_store_4d(const void* tmap, uint32_t src, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(tmap),
                 "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
template <int N> __device__ __forceinline__ void bulk_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_leader(uint32_t bar) {   // arrive on the pair leader's barrier
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(bar & PEER_MASK) : "memory");
}
template <bool kTwoCta> __device__ __forceinline__ void tmem_alloc_t(uint32_t smem_dst, uint32_t ncols) {
    if (kTwoCta) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
        ptx::tmem_alloc(smem_dst, ncols);
        ptx::tmem_relinquish();
    }
}
template <bool kTwoCta> __device__ __forceinline__ void tmem_dealloc_t(uint32_t taddr, uint32_t ncols) {
    if (kTwoCta)
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
    else
        ptx::tmem_dealloc(taddr, ncols);
}
template <bool kTwoCta>
__device__ __forceinline__ void mma_t(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                      uint32_t accumulate) {
    if (kTwoCta) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "setp.ne.b32 p, %4, 0;\n"
            "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
            "}\n" ::"r"(d_tmem),
            "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
            : "memory");
    } else {
        ptx::mma_ss(d_tmem, a_desc, b_desc, idesc, accumulate);
    }
}
// mbarrier arrive once the MMAs issued so far have completed; pair mode: on this barrier in BOTH CTAs
template <bool kTwoCta> __device__ __forceinline__ void commit_t(uint32_t bar) {
    if (kTwoCta) {
        asm volatile(
            "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                bar),
            "h"((uint16_t)0x3)
            : "memory");
    } else {
        ptx::tc_commit(bar);
    }
}
__device__ __forceinline__ void named_bar_sync(int id, int threads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}
__device__ __forceinline__ Vec16 lds16(uint32_t addr) {
    Vec16 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.w[0]), "=r"(v.w[1]), "=r"(v.w[2]), "=r"(v.w[3]) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts16(uint32_t addr, const Vec16& v) {
    asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(v.w[0]), "r"(v.w[1]), "r"(v.w[2]), "r"(v.w[3])
                 : "memory");
}
__device__ __forceinline__ Vec16 ldg16_nc(const void* p) {
    Vec16 v;
    asm volatile("ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.w[0]), "=r"(v.w[1]), "=r"(v.w[2]), "=r"(v.w[3]) : "l"(p));
    return v;
}

// f[0..7] += the eight 16-bit values of v.  bf16 -> fp32 is a shift (low half) or a mask (high half): two integer
// instructions per pair instead of the three the generic element-wise conversion compiles to.
template <typename T>
__device__ __forceinline__ void add8(float (&f)[8], const Vec16& v) {
    if constexpr (std::is_same<T, __nv_bfloat16>::value) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            f[2 * i] += __uint_as_float(v.w[i] << 16);
            f[2 * i + 1] += __uint_as_float(v.w[i] & 0xffff0000u);
        }
    } else {
        float t[8];
        unpack8<T>(v, t);
#pragma unroll
        for (int i = 0; i < 8; ++i) f[i] += t[i];
    }
}

// x -> 0.5 x (1 + erf(x / sqrt 2)): exact GELU (torch.nn.functional.gelu default).  erf by Abramowitz-Stegun 7.1.26
// (|error| <= 1.5e-7, far below the 16-bit rounding of the product): one reciprocal, one exp2, a degree-5 Horner.
__device__ __forceinline__ float gelu_erf(float x) {
    const float t = fabsf(x) * 0.70710678118654752f;
    float k;   // rcp.approx (1 ulp): the IEEE-rounded reciprocal costs a slow-path call per element
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(k) : "f"(fmaf(0.3275911f, t, 1.0f)));
    float p = fmaf(1.061405429f, k, -1.453152027f);
    p = fmaf(p, k, 1.421413741f);
    p = fmaf(p, k, -0.284496736f);
    p = fmaf(p, k, 0.254829592f);
    const float e = ptx::ex2_approx(-1.4426950408889634f * t * t);
    const float erf_abs = fmaf(-p * k, e, 1.0f);         // erf(|x| / sqrt 2)
    return 0.5f * x + 0.5f * fabsf(x) * erf_abs;          // 0.5 x (1 + sign(x) erf(|x| / sqrt 2))
}

// The same for a pair of gates on the packed fp32x2 pipe (FFMA2 / FMUL2: two lanes per issue slot) — the GEGLU
// epilogue is bounded by instruction issue, and 12 of gelu_erf's 16 arithmetic instructions are FMA-class.
// v2 (a pair of values) is multiplied by gelu(g2) and returned.
__device__ __forceinline__ uint64_t mul_gelu_erf2(uint64_t v2, uint64_t g2) {
    float g0, g1;
    ptx::unpack2(g2, g0, g1);
    const uint64_t ax = ptx::pack2(fabsf(g0), fabsf(g1));
    const uint64_t t = ptx::mul2(ax, ptx::pack2(0.70710678118654752f, 0.70710678118654752f));
    const uint64_t d = ptx::fma2(ptx::pack2(0.3275911f, 0.3275911f), t, ptx::pack2(1.0f, 1.0f));
    float d0, d1, k0, k1;
    ptx::unpack2(d, d0, d1);
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(k0) : "f"(d0));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(k1) : "f"(d1));
    const uint64_t k = ptx::pack2(k0, k1);
    uint64_t p = ptx::fma2(ptx::pack2(1.061405429f, 1.061405429f), k, ptx::pack2(-1.453152027f, -1.453152027f));
    p = ptx::fma2(p, k, ptx::pack2(1.421413741f, 1.421413741f));
    p = ptx::fma2(p, k, ptx::pack2(-0.284496736f, -0.284496736f));
    p = ptx::fma2(p, k, ptx::pack2(0.254829592f, 0.254829592f));
    const uint64_t ea = ptx::mul2(ptx::mul2(t, t), ptx::pack2(-1.4426950408889634f, -1.4426950408889634f));
    float e0, e1;
    ptx::unpack2(ea, e0, e1);
    const uint64_t e = ptx::pack2(ptx::ex2_approx(e0), ptx::ex2_approx(e1));
    const uint64_t erf_abs = ptx::sub2(ptx::pack2(1.0f, 1.0f), ptx::mul2(ptx::mul2(p, k), e));   // erf(|g| / sqrt 2)
    const uint64_t half = ptx::pack2(0.5f, 0.5f);
    const uint64_t gelu = ptx::fma2(ptx::mul2(ax, half), erf_abs, ptx::mul2(g2, half));
    return ptx::mul2(v2, gelu);
}

struct TileCoord {
    int n_tile, c1, c2, c3;
};

template <typename C>
__device__ __forceinline__ TileCoord decode_tile(const Params& p, int t, uint32_t crank) {
    TileCoord tc;
    tc.n_tile = t % p.n_tiles;
    int m = t / p.n_tiles;
    if (C::kTwoCta) m = 2 * m + (int)crank;
    const int i1 = m % p.t1;
    m /= p.t1;
    const int i2 = m % p.t2;
    const int i3 = m / p.t2;            // may run past the tensor for the padding tile of an odd pair: all OOB
    tc.c1 = i1 * p.b1;
    tc.c2 = i2 * p.b2;
    tc.c3 = i3 * p.b3;
    return tc;
}

// accumulator columns in use for column tile n_tile
template <typename C>
__device__ __forceinline__ int tile_cols(const Params& p, int n_tile) {
    if (C::kEpi != EPI_GEGLU && p.tail_cols > 0 && n_tile == p.n_tiles - 1) return p.tail_cols;
    return C::BN;
}

template <typename C, typename T>
__global__ void __launch_bounds__(C::THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tm_a0, const __grid_constant__ CUtensorMap tm_w0,
               const __grid_constant__ CUtensorMap tm_a1, const __grid_constant__ CUtensorMap tm_w1,
               const __grid_constant__ CUtensorMap tm_out, const __grid_constant__ CUtensorMap tm_res,
               const __grid_constant__ Params prm) {   // __grid_constant__: the dynamically indexed tap table is read
                                                       // from the constant bank instead of a per-thread local copy
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const uint32_t sbase = smem_u32(smem_raw);
    MVOC_REQUIRE_SMEM_1024(sbase, "gemm_tc_kernel");
    constexpr int kStages = C::kStages;
    constexpr int N_OUT = C::N_OUT;
    const uint32_t sOut = sbase + C::out_off;
    const uint32_t sStage = sbase + C::stage_off;
    const uint32_t bars = sbase + C::bar_off;
    const uint32_t b_full = bars, b_empty = bars + 8 * kStages, b_acc_full = bars + 16 * kStages,
                   b_acc_empty = b_acc_full + 16, b_res = b_acc_empty + 16;
    const uint32_t s_tmem_ptr = sbase + C::tmem_ptr_off;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t crank = C::kTwoCta ? cluster_ctarank() : 0u;
    const bool leader = crank == 0;
    const int first_tile = C::kTwoCta ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
    const int tile_stride = C::kTwoCta ? (int)(gridDim.x >> 1) : (int)gridDim.x;

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tensormap(&tm_a0);
        ptx::prefetch_tensormap(&tm_w0);
        ptx::prefetch_tensormap(&tm_out);
        if (prm.n_src > 1) {
            ptx::prefetch_tensormap(&tm_a1);
            ptx::prefetch_tensormap(&tm_w1);
        }
        if (prm.has_res) ptx::prefetch_tensormap(&tm_res);
        for (int s = 0; s < kStages; ++s) {
            ptx::mbar_init(b_full + 8 * s, 1);
            ptx::mbar_init(b_empty + 8 * s, 1);
        }
        for (int b = 0; b < 2; ++b) {
            ptx::mbar_init(b_acc_full + 8 * b, 1);
            ptx::mbar_init(b_acc_empty + 8 * b, (C::kTwoCta ? 2 : 1) * C::EPI_WARPS);   // one arrive per epilogue warp (of both CTAs)
        }
        for (int b = 0; b < C::EPI_WARPS * N_OUT; ++b) ptx::mbar_init(b_res + 8 * b, 1);
        ptx::fence_mbar_init();
    }
    if (warp == 1) tmem_alloc_t<C::kTwoCta>(s_tmem_ptr, TMEM_COLS);
    ptx::tc_fence_before();
    __syncthreads();
    if (C::kTwoCta) cluster_sync_all();   // the peer's barriers exist before anything is signalled on them
    ptx::tc_fence_after();
    const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(smem_raw + C::tmem_ptr_off);

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            uint32_t it = 0;
            for (int t = first_tile; t < prm.total_tiles; t += tile_stride) {
                const TileCoord tc = decode_tile<C>(prm, t, crank);
                for (int src = 0; src < prm.n_src; ++src) {
                    const CUtensorMap* ma = src ? &tm_a1 : &tm_a0;
                    const CUtensorMap* mw = src ? &tm_w1 : &tm_w0;
                    const int taps = prm.taps[src];
                    for (int kc = 0; kc < prm.k_chunks[src]; ++kc)
                        for (int tap = 0; tap < taps; ++tap, ++it) {   // taps innermost: shifted boxes share L2 lines
                            const uint32_t s = it % kStages;
                            const uint32_t ph = (it / kStages) & 1u;
                            ptx::mbar_wait(b_empty + 8 * s, ph ^ 1u, 1);
                            const uint32_t sA = sStage + s * C::STAGE_BYTES, sB = sA + A_BYTES;
                            const uint32_t full = b_full + 8 * s;
                            const bool skip_w = (prm.dbg & 1) && it >= (uint32_t)kStages;
                            const bool skip_a = (prm.dbg & 2) && it >= (uint32_t)kStages;
                            const uint32_t bytes = (skip_a ? 0 : A_BYTES) + (skip_w ? 0 : C::B_BYTES);
                            if (!C::kTwoCta) ptx::mbar_expect_tx(full, bytes);
                            else if (leader) ptx::mbar_expect_tx(full, 2 * bytes);
                            if (!skip_a)
                                tma_load_tile<C::kTwoCta>(sA, ma, full, kc * KC,
                                                          prm.a_stride * tc.c1 + prm.off[src][tap][0],
                                                          prm.a_stride * tc.c2 + prm.off[src][tap][1],
                                                          tc.c3 + prm.off[src][tap][2]);
                            if (skip_w) continue;
                            if (C::kEpi == EPI_GEGLU) {
                                // accumulator columns = NP value columns then NP gate columns of the same Linear
                                constexpr int NP = C::BN / 2;
                                if (C::kTwoCta) {   // leader stages the value rows, the peer the gate rows
                                    const int wrow = tc.n_tile * NP + (leader ? 0 : prm.gate_off);
                                    tma_load_tile<true>(sB, mw, full, kc * KC, wrow, tap, 0);
                                } else {
                                    tma_load_tile<false>(sB, mw, full, kc * KC, tc.n_tile * NP, tap, 0);
                                    tma_load_tile<false>(sB + NP * KC * 2, mw, full, kc * KC,
                                                         tc.n_tile * NP + prm.gate_off, tap, 0);
                                }
                            } else {
                                // pair mode: this CTA stages its half of the tile's weight rows (a narrower tail tile
                                // still loads a full box: the rows beyond the tail are never read by its MMAs)
                                const int wrow = tc.n_tile * C::BN +
                                                 (C::kTwoCta ? (int)crank * (tile_cols<C>(prm, tc.n_tile) / 2) : 0);
                                tma_load_tile<C::kTwoCta>(sB, mw, full, kc * KC, wrow, tap, 0);
                            }
                        }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (pair mode: the leader CTA only) =====================
        if (lane == 0 && leader) {
            constexpr bool kF16 = sizeof(T) == 2 && !std::is_same<T, __nv_bfloat16>::value;
            uint32_t it = 0, lt = 0;
            for (int t = first_tile; t < prm.total_tiles; t += tile_stride, ++lt) {
                const uint32_t IDESC =
                    ptx::idesc_f16(kF16, C::kTwoCta ? 256 : 128, tile_cols<C>(prm, t % prm.n_tiles), false);
                const uint32_t buf = lt & 1u;
                ptx::mbar_wait(b_acc_empty + 8 * buf, ((lt >> 1) & 1u) ^ 1u, 2);
                ptx::tc_fence_after();
                const uint32_t tacc = tmem + buf * C::BN;
                int n_chunks = 0;
                for (int src = 0; src < prm.n_src; ++src) n_chunks += prm.k_chunks[src] * prm.taps[src];
                for (int c = 0; c < n_chunks; ++c, ++it) {
                    const uint32_t s = it % kStages;
                    const uint32_t ph = (it / kStages) & 1u;
                    ptx::mbar_wait(b_full + 8 * s, ph, 3);
                    ptx::tc_fence_after();
                    const uint32_t sA = sStage + s * C::STAGE_BYTES, sB = sA + A_BYTES;
                    const uint64_t a0 = ptx::smem_desc_sw128(sA, 16, 1024);
                    const uint64_t b0 = ptx::smem_desc_sw128(sB, 16, 1024);
#pragma unroll
                    for (int ks = 0; ks < KC / 16; ++ks)   // +32 B per 16-element K step (encoded >> 4)
                        mma_t<C::kTwoCta>(tacc, a0 + (uint64_t)(ks * 2), b0 + (uint64_t)(ks * 2), IDESC,
                                          (c > 0 || ks > 0) ? 1u : 0u);
                    commit_t<C::kTwoCta>(b_empty + 8 * s);   // stage reusable once these MMAs have read it
                }
                commit_t<C::kTwoCta>(b_acc_full + 8 * buf);   // accumulator complete (both CTAs in pair mode)
            }
        }
    } else {
        // ===================== epilogue (warps 2-9), one independent pipeline per warp =====================
        // Warp q owns rows [32q, 32q+32) of the tile (the TMEM lanes it may read).  Per slab of SLAB columns:
        // tcgen05.ld (issued one slab ahead) -> + bias -> (+ residual, TMA-loaded into the staging buffer two slabs
        // ahead) -> (GEGLU) -> 16-bit -> swizzled staging -> TMA store of the warp's own 32-row box.  No barrier
        // wider than the warp: lane 0 owns the warp's bulk-async groups and residual barriers.
        constexpr int SLAB = C::SLAB, SLABS = C::SLABS;
        constexpr int CHUNKS = SLAB / 8;                    // 16-byte chunks per staged row
        constexpr int HALVES = C::HALVES;
        const int q = warp & 3;              // TMEM lane quarter this warp may read (hardware: warp id % 4)
        const int ew = warp - 2;             // epilogue warp index
        const int half = ew >> 2;            // which of the HALVES interleaved slab sequences this warp takes
        const int my_slabs = (SLABS - half + HALVES - 1) / HALVES;   // slabs half, half + HALVES, ... of every tile
        const uint32_t sWarp = sOut + (uint32_t)ew * (N_OUT * C::WSLAB_BYTES);
        const uint32_t row_off = (uint32_t)lane * (SLAB * 2);
        // swizzle of the staging rows (what the TMA store expects): 128B -> chunk ^ (row & 7); 64B -> chunk ^ ((row >> 1) & 3)
        const uint32_t sw = SLAB == 64 ? (uint32_t)(lane & 7) : (uint32_t)((lane >> 1) & 3);
        const uint32_t b_res_w = b_res + 8 * (ew * N_OUT);
        const T* bias = reinterpret_cast<const T*>(prm.bias);
        // rows 32q.. of the tile inside the (b1, b2, b3) row box
        const int r0 = q * 32;
        const int w1 = r0 % prm.b1, w2 = (r0 / prm.b1) % prm.b2, w3 = r0 / (prm.b1 * prm.b2);

        auto slab_at = [&](uint32_t g, int& col, TileCoord& tc) -> bool {   // slab g of this warp -> column, row coords
            const int t = first_tile + (int)(g / my_slabs) * tile_stride;
            if (t >= prm.total_tiles) return false;
            tc = decode_tile<C>(prm, t, crank);
            col = tc.n_tile * C::OUT_COLS + ((int)(g % my_slabs) * HALVES + half) * SLAB;
            return true;
        };
        auto prefetch_res = [&](uint32_t g) {   // lane 0 only
            int col;
            TileCoord tc;
            if (!slab_at(g, col, tc)) return;
            const uint32_t ob = g % N_OUT;
            ptx::mbar_expect_tx(b_res_w + 8 * ob, C::WSLAB_BYTES);
            ptx::tma_load_4d(sWarp + ob * C::WSLAB_BYTES, &tm_res, b_res_w + 8 * ob, col, tc.c1 + w1, tc.c2 + w2,
                             tc.c3 + w3);
        };
        if (lane == 0 && prm.has_res)
            for (int a = 0; a < C::RES_AHEAD; ++a) prefetch_res(a);
        uint32_t g = 0, lt = 0;
        for (int t = first_tile; t < prm.total_tiles; t += tile_stride, ++lt) {
            const TileCoord tc = decode_tile<C>(prm, t, crank);
            const uint32_t buf = lt & 1u;
            ptx::mbar_wait(b_acc_full + 8 * buf, (lt >> 1) & 1u, 4);
            ptx::tc_fence_after();
            const uint32_t tacc = tmem + ((uint32_t)(q * 32) << 16) + buf * C::BN;
            const int col0 = tc.n_tile * C::OUT_COLS;
            if ((prm.dbg & 8) && !prm.has_res) {   // experiment: how fast is the kernel without its epilogue
                ptx::tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    if (C::kTwoCta) mbar_arrive_leader(b_acc_empty + 8 * buf);
                    else ptx::mbar_arrive(b_acc_empty + 8 * buf);
                }
                continue;
            }
            uint32_t r[2][SLAB];                               // value columns, two slabs in flight
            uint32_t gt[C::kEpi == EPI_GEGLU ? SLAB : 1];      // gate columns (GEGLU)
            auto issue_ld = [&](int sl, int which) {
#pragma unroll
                for (int c = 0; c < SLAB / 32; ++c)
                    ptx::tmem_ld32(tacc + sl * SLAB + c * 32, *reinterpret_cast<uint32_t(*)[32]>(&r[which][c * 32]));
                if constexpr (C::kEpi == EPI_GEGLU)
                    ptx::tmem_ld32(tacc + C::BN / 2 + sl * SLAB, *reinterpret_cast<uint32_t(*)[32]>(&gt[0]));
            };
            auto release_acc = [&]() {                       // accumulator buffer drained: back to the MMA warp
                ptx::tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    if (C::kTwoCta) mbar_arrive_leader(b_acc_empty + 8 * buf);
                    else ptx::mbar_arrive(b_acc_empty + 8 * buf);
                }
            };
            auto process = [&](int sl, const uint32_t (&acc)[SLAB]) {
                const uint32_t ob = g % N_OUT;
                const uint32_t sbuf = sWarp + ob * C::WSLAB_BYTES + row_off;
                if (prm.has_res) ptx::mbar_wait(b_res_w + 8 * ob, (g / N_OUT) & 1u, 5);
#pragma unroll
                for (int c = 0; c < CHUNKS; ++c) {
                    float f[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) f[e] = __uint_as_float(acc[c * 8 + e]);
                    if (bias) add8<T>(f, ldg16_nc(bias + col0 + sl * SLAB + c * 8));
                    if constexpr (C::kEpi == EPI_GEGLU) {
                        float gv[8];
#pragma unroll
                        for (int e = 0; e < 8; ++e) gv[e] = __uint_as_float(gt[c * 8 + e]);
                        if (bias) add8<T>(gv, ldg16_nc(bias + prm.gate_off + col0 + sl * SLAB + c * 8));
#pragma unroll
                        for (int e = 0; e < 8; e += 2)
                            ptx::unpack2(mul_gelu_erf2(ptx::pack2(f[e], f[e + 1]), ptx::pack2(gv[e], gv[e + 1])), f[e],
                                         f[e + 1]);
                    }
                    if constexpr (C::kEpi == EPI_GELU) {   // gelu(acc + bias) = 1 x gelu(acc + bias): the GEGLU gate code
#pragma unroll
                        for (int e = 0; e < 8; e += 2)
                            ptx::unpack2(mul_gelu_erf2(ptx::pack2(1.0f, 1.0f), ptx::pack2(f[e], f[e + 1])), f[e], f[e + 1]);
                    }
                    const uint32_t addr = sbuf + (((uint32_t)c ^ sw) << 4);
                    if (prm.has_res) add8<T>(f, lds16(addr));
                    sts16(addr, pack8<T>(f));
                }
                ptx::fence_proxy_async_smem();          // generic-proxy writes -> visible to the TMA store
                __syncwarp();
                if (lane == 0) {
                    if (!(prm.dbg & 4))
                        tma_store_4d(&tm_out, sWarp + ob * C::WSLAB_BYTES, col0 + sl * SLAB, tc.c1 + w1, tc.c2 + w2, tc.c3 + w3);
                    ptx::bulk_commit();
                    bulk_wait_read<C::ST_PENDING>();     // stores up to slab g - ST_PENDING have released their buffers
                    if (prm.has_res) prefetch_res(g + C::RES_AHEAD);   // into the buffer slab g - ST_PENDING used
                }
                ++g;
            };
            if constexpr (C::kEpi == EPI_GEGLU) {
                // the gate makes this epilogue compute-heavy (one erf per output): keep the code small (no unrolling
                // across slabs: the unrolled form overflowed the instruction cache and ran 1.7x slower on B200)
#pragma unroll 1
                for (int i = 0; i < my_slabs; ++i) {
                    const int sl = i * HALVES + half;
                    issue_ld(sl, 0);
                    ptx::tmem_wait_ld();
                    if (i + 1 == my_slabs) release_acc();
                    process(sl, r[0]);
                }
            } else {
                const int width = tile_cols<C>(prm, tc.n_tile);   // < BN for the tail tile only
                constexpr int MAX_W = (SLABS + HALVES - 1) / HALVES;
                if (half * SLAB < width) issue_ld(half, 0);
#pragma unroll
                for (int i = 0; i < MAX_W; ++i) {
                    if (i < my_slabs) {                          // warp-uniform
                        const int sl = i * HALVES + half;
                        ptx::tmem_wait_ld();                     // slab sl is in r[i & 1]
                        if (i + 1 < my_slabs) {
                            if ((sl + HALVES) * SLAB < width) issue_ld(sl + HALVES, (i & 1) ^ 1);   // streams in meanwhile
                        } else {
                            release_acc();
                        }
                        if (sl * SLAB < width) {
                            process(sl, r[i & 1]);
                        } else {
                            // slab beyond the tail tile: no columns, but the buffer rotation, the residual barrier
                            // phases and the bulk-group count stay those of a full tile
                            const uint32_t ob = g % N_OUT;
                            if (prm.has_res) ptx::mbar_wait(b_res_w + 8 * ob, (g / N_OUT) & 1u, 5);
                            __syncwarp();
                            if (lane == 0) {
                                ptx::bulk_commit();
                                bulk_wait_read<C::ST_PENDING>();
                                if (prm.has_res) prefetch_res(g + C::RES_AHEAD);
                            }
                            ++g;
                        }
                    }
                }
            }
        }
        if (lane == 0) bulk_wait_all();
        ptx::tc_fence_before();
    }

    __syncthreads();
    if (C::kTwoCta) cluster_sync_all();   // neither CTA leaves (or frees TMEM) while its peer may still use it
    if (warp == 1) {
        ptx::tc_fence_after();
        tmem_dealloc_t<C::kTwoCta>(tmem, TMEM_COLS);
    }
}

// ------------------------------------------------------------------ host ---
// Row box (b1, b2, b3), powers of two with product 128, that wastes the fewest zero-filled rows on the
// (d1, d2, d3) grid; ties go to the widest box along d1 (longest contiguous runs).
static void choose_box(int64_t d1, int64_t d2, int64_t d3, int* b1, int* b2, int* b3) {
    int64_t best = -1;
    for (int w = 128; w >= 1; w >>= 1)
        for (int h = 128 / w; h >= 1; h >>= 1) {
            const int n = 128 / (w * h);
            const int64_t padded = ((d1 + w - 1) / w) * w * ((d2 + h - 1) / h) * h * ((d3 + n - 1) / n) * n;
            if (best < 0 || padded < best) {
                best = padded;
                *b1 = w, *b2 = h, *b3 = n;
            }
        }
}

// One (activation, weight) source of the K loop.
struct Source {
    const void* a;
    int64_t K;                 // channels (multiple of 64)
    int64_t a_dim[3];          // extents of the activation along d1, d2, d3 (the row grid unless stride > 1)
    int64_t a_str[3];          // element strides of d1, d2, d3
    int stride;                // 1, or 2 for a stride-2 convolution (every source of a problem shares it)
    const void* w;             // [taps, n_rows, K] contiguous
    int taps;
    int8_t off[MAX_TAPS][3];
};

struct Problem {
    int dtype;
    int64_t d1, d2, d3;        // row grid
    int n_src;
    Source src[2];
    int64_t N;                 // output columns (GEGLU: F)
    int64_t w_rows;            // rows of each weight tap (N, GEGLU: 2F)
    const void* bias;
    const void* residual;
    int64_t res_str[3];
    void* out;
    int64_t out_str[3];
    int geglu;
    int gelu;                  // exact GELU on the Linear's output (EPI_GELU)
    int variant;               // bit 0: CTA pairs; bit 1: no tail tiles; bits 8..16: BN override (0 = auto)
    const char* what;
};

template <typename C, typename T>
static int launch_cfg(const Problem& pb, Params prm, int b1, int b2, int b3, cudaStream_t stream) {
    const char* what = pb.what;
    static bool smem_set[64] = {false};
    int rc = set_max_dynamic_smem((const void*)gemm_tc_kernel<C, T>, C::alloc, smem_set, what);
    if (rc != MVOC_OK) return rc;
    CUtensorMap ma[2], mw[2], mo, mr;
    for (int s = 0; s < pb.n_src; ++s) {
        const Source& sc = pb.src[s];
        const int64_t dims[4] = {sc.K, sc.a_dim[0], sc.a_dim[1], sc.a_dim[2]};
        const int box[4] = {KC, b1 * sc.stride, b2 * sc.stride, b3};
        if ((rc = make_map4(&ma[s], sc.a, pb.dtype, dims, sc.a_str, box, sc.stride, CU_TENSOR_MAP_SWIZZLE_128B,
                            what, s ? "x2" : "x")) != MVOC_OK)
            return rc;
        const int64_t wd[4] = {sc.K, pb.w_rows, sc.taps, 1};
        const int64_t ws[3] = {sc.K, sc.K * pb.w_rows, sc.K * pb.w_rows * sc.taps};
        const int wb[4] = {KC, C::kEpi == EPI_GEGLU ? C::BN / 2 : C::B_ROWS, 1, 1};
        if ((rc = make_map4(&mw[s], sc.w, pb.dtype, wd, ws, wb, 1, CU_TENSOR_MAP_SWIZZLE_128B, what,
                            s ? "w2" : "w")) != MVOC_OK)
            return rc;
    }
    if (pb.n_src == 1) ma[1] = ma[0], mw[1] = mw[0];
    {
        // the epilogue stores per warp: a box of 32 rows (the first 32 rows of the row box) x SLAB columns
        const int sb1 = b1 < 32 ? b1 : 32, sb2 = b2 < 32 / sb1 ? b2 : 32 / sb1, sb3 = 32 / (sb1 * sb2);
        const int64_t dims[4] = {pb.N, pb.d1, pb.d2, pb.d3};
        const int box[4] = {C::SLAB, sb1, sb2, sb3};
        const CUtensorMapSwizzle swz = C::SLAB == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
        if ((rc = make_map4(&mo, pb.out, pb.dtype, dims, pb.out_str, box, 1, swz, what, "out")) != MVOC_OK) return rc;
        if (pb.residual) {
            if ((rc = make_map4(&mr, pb.residual, pb.dtype, dims, pb.res_str, box, 1, swz, what, "residual")) !=
                MVOC_OK)
                return rc;
        } else {
            mr = mo;
        }
    }
    prm.n_tiles = (int)((pb.N + C::OUT_COLS - 1) / C::OUT_COLS);
    prm.tail_cols = (int)(pb.N % C::OUT_COLS);
    MVOC_REQUIRE(prm.tail_cols == 0 || (C::kEpi != EPI_GEGLU && prm.tail_cols % 64 == 0),
                 MVOC_ERR_UNSUPPORTED, "%s: N=%lld does not tile by %d columns", what, (long long)pb.N, C::OUT_COLS);
    const int64_t m_tiles = (int64_t)prm.t1 * prm.t2 * ((pb.d3 + b3 - 1) / b3);
    const int64_t units = C::kTwoCta ? (m_tiles + 1) / 2 : m_tiles;
    const int64_t total = units * prm.n_tiles;
    MVOC_REQUIRE(total > 0 && total <= 0x7fffffffLL, MVOC_ERR_UNSUPPORTED, "%s: %lld tiles", what, (long long)total);
    prm.total_tiles = (int)total;
    const int sms = num_sms();
    int64_t ctas = C::kTwoCta ? 2 * (total < sms / 2 ? total : sms / 2) : (total < sms ? total : sms);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)ctas);
    cfg.blockDim = dim3(C::THREADS);
    cfg.dynamicSmemBytes = C::alloc;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = C::kTwoCta ? 2 : 1;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, gemm_tc_kernel<C, T>, ma[0], mw[0], ma[1], mw[1], mo, mr, prm);
    MVOC_REQUIRE(e == cudaSuccess, MVOC_ERR_CUDA, "%s: launch failed: %s", what, cudaGetErrorString(e));
    return MVOC_OK;
}

template <int BN, int kEpi>
static int launch_bn(const Problem& pb, const Params& prm, int b1, int b2, int b3, cudaStream_t s, bool two) {
    if (pb.dtype == MVOC_F16) {
        if (two) return launch_cfg<Cfg<BN, true, kEpi>, __half>(pb, prm, b1, b2, b3, s);
        return launch_cfg<Cfg<BN, false, kEpi>, __half>(pb, prm, b1, b2, b3, s);
    }
    if (two) return launch_cfg<Cfg<BN, true, kEpi>, __nv_bfloat16>(pb, prm, b1, b2, b3, s);
    return launch_cfg<Cfg<BN, false, kEpi>, __nv_bfloat16>(pb, prm, b1, b2, b3, s);
}

// Tile width (0 = none fits) and CTA mode for a problem of m_tiles 128-row tiles x N output columns on a chip of `sms`
// SMs: the cheapest of waves x chunk cost over the available widths.  variant bit 0 allows CTA pairs, bit 1 forbids a
// narrower tail tile, bits 8.. force a width.  Also exported as mvoc_gemm_plan (host logic, testable without a GPU).
static void plan_tiles(int64_t m_tiles, int64_t N, bool geglu, int variant, int sms, int* bn_out, bool* pair_out) {
    const int forced = (variant >> 8) & 0x1ff;
    const bool allow_pair = (variant & 1) != 0;
    const int widths_lin[5] = {256, 192, 160, 128, 64};
    const int widths_geglu[2] = {256, 128};
    const int* widths = geglu ? widths_geglu : widths_lin;
    const int n_widths = geglu ? 2 : 5;
    const bool allow_tail = (variant & 2) == 0;   // variant bit 1: only widths that divide N (A/B switch)
    int BN = 0;
    bool two = false;
    double best = 0.0;
    for (int i = 0; i < n_widths; ++i) {
        const int w = widths[i];
        const int out_cols = geglu ? w / 2 : w;
        if (forced && forced != w) continue;
        // a narrower LAST column tile (multiple of 64 columns) lets 256-wide tiles cover N = 640, 1920, 320 ...
        const int tail = (int)(N % out_cols);
        if (tail != 0 && (geglu || !allow_tail || w % 64 != 0 || tail % 64 != 0)) continue;
        const int64_t n_full = N / out_cols;
        const int64_t n_tiles = n_full + (tail ? 1 : 0);
        for (int pair = allow_pair ? 1 : 0; pair >= 0; --pair) {
            const int64_t units = (pair ? (m_tiles + 1) / 2 : m_tiles) * n_tiles;
            const int64_t slots = pair ? sms / 2 : sms;
            const double waves = (double)((units + slots - 1) / slots);
            // a pair tile covers two row tiles; the tail tile still fills a full-width weight box
            const double per_tile = ((double)n_full * chunk_cost(w, pair != 0) +
                                     (tail ? 0.5 * (chunk_cost(tail, pair != 0) + chunk_cost(w, pair != 0)) : 0.0)) /
                                    (double)n_tiles;
            const double cost = waves * per_tile;
            if (BN == 0 || cost < best * 0.999) best = cost, BN = w, two = pair != 0;
        }
    }
    *bn_out = BN;
    *pair_out = two;
}

static int run(const Problem& pb, cudaStream_t stream) {
    const char* what = pb.what;
    MVOC_REQUIRE(pb.dtype == MVOC_BF16 || pb.dtype == MVOC_F16, MVOC_ERR_UNSUPPORTED,
                 "%s: dtype %d unsupported (bf16 / fp16)", what, pb.dtype);
    MVOC_REQUIRE(pb.d1 > 0 && pb.d2 > 0 && pb.d3 > 0, MVOC_ERR_INVALID_ARG, "%s: empty row grid %lld x %lld x %lld", what,
                 (long long)pb.d1, (long long)pb.d2, (long long)pb.d3);
    MVOC_REQUIRE(pb.d1 <= 0x7fffffffLL && pb.d2 <= 0x7fffffffLL && pb.d3 <= 0x7fffffffLL, MVOC_ERR_UNSUPPORTED,
                 "%s: row grid too large", what);
    MVOC_REQUIRE(pb.N > 0 && pb.N % 64 == 0, MVOC_ERR_UNSUPPORTED, "%s: N=%lld must be a multiple of 64", what,
                 (long long)pb.N);
    MVOC_REQUIRE(pb.out != nullptr && (uintptr_t)pb.out % 16 == 0 && (uintptr_t)pb.bias % 16 == 0 &&
                     (uintptr_t)pb.residual % 16 == 0,
                 MVOC_ERR_INVALID_ARG, "%s: out / bias / residual must be non-null (out) and 16-byte aligned", what);
    Params prm{};
    prm.n_src = pb.n_src;
    for (int s = 0; s < pb.n_src; ++s) {
        const Source& sc = pb.src[s];
        MVOC_REQUIRE(sc.a && sc.w && (uintptr_t)sc.a % 16 == 0 && (uintptr_t)sc.w % 16 == 0, MVOC_ERR_INVALID_ARG,
                     "%s: activation / weight pointers must be non-null and 16-byte aligned", what);
        MVOC_REQUIRE(sc.K > 0 && sc.K % 64 == 0, MVOC_ERR_UNSUPPORTED, "%s: K=%lld must be a multiple of 64", what,
                     (long long)sc.K);
        MVOC_REQUIRE(sc.taps >= 1 && sc.taps <= MAX_TAPS, MVOC_ERR_INVALID_ARG, "%s: %d taps", what, sc.taps);
        MVOC_REQUIRE(sc.stride == pb.src[0].stride && (sc.stride == 1 || sc.stride == 2), MVOC_ERR_UNSUPPORTED,
                     "%s: activation stride %d (1 or 2, the same for every source)", what, sc.stride);
        prm.k_chunks[s] = (int)(sc.K / 64);
        prm.taps[s] = sc.taps;
        for (int t = 0; t < sc.taps; ++t)
            for (int d = 0; d < 3; ++d) prm.off[s][t][d] = sc.off[t][d];
    }
    int b1, b2, b3;
    choose_box(pb.d1, pb.d2, pb.d3, &b1, &b2, &b3);
    prm.b1 = b1, prm.b2 = b2, prm.b3 = b3;
    prm.t1 = (int)((pb.d1 + b1 - 1) / b1);
    prm.t2 = (int)((pb.d2 + b2 - 1) / b2);
    prm.bias = pb.bias;
    prm.has_res = pb.residual != nullptr;
    prm.a_stride = pb.src[0].stride;
    prm.gate_off = (int)pb.N;
    prm.dbg = (pb.variant >> 20) & 15;
    // Tile width and CTA mode.  Wide tiles win (chunk_cost above) — until the problem has fewer tiles than the chip
    // has SMs (the low-resolution levels, and every level once the frames are sharded over 8 GPUs), where narrower
    // tiles and single CTAs fill more SMs.  Pick the cheapest of
    // waves x chunk cost; variant bit 0 allows CTA pairs, bit 1 forbids a narrower tail tile, bits 8.. force a width.
    const int64_t m_tiles = (int64_t)prm.t1 * prm.t2 * ((pb.d3 + b3 - 1) / b3);
    const int forced = (pb.variant >> 8) & 0x1ff;
    int BN = 0;
    bool two = false;
    plan_tiles(m_tiles, pb.N, pb.geglu != 0, pb.variant, num_sms(), &BN, &two);
    MVOC_REQUIRE(BN != 0, MVOC_ERR_UNSUPPORTED, "%s: no tile width (forced %d) divides N=%lld", what, forced,
                 (long long)pb.N);
    if (pb.geglu) {
        if (BN == 256) return launch_bn<256, EPI_GEGLU>(pb, prm, b1, b2, b3, stream, two);
        return launch_bn<128, EPI_GEGLU>(pb, prm, b1, b2, b3, stream, two);
    }
    if (pb.gelu) {
        switch (BN) {
            case 256: return launch_bn<256, EPI_GELU>(pb, prm, b1, b2, b3, stream, two);
            case 192: return launch_bn<192, EPI_GELU>(pb, prm, b1, b2, b3, stream, two);
            case 160: return launch_bn<160, EPI_GELU>(pb, prm, b1, b2, b3, stream, two);
            case 128: return launch_bn<128, EPI_GELU>(pb, prm, b1, b2, b3, stream, two);
            case 64: return launch_bn<64, EPI_GELU>(pb, prm, b1, b2, b3, stream, two);
            default: break;
        }
    }
    switch (BN) {
        case 256: return launch_bn<256, EPI_LINEAR>(pb, prm, b1, b2, b3, stream, two);
        case 192: return launch_bn<192, EPI_LINEAR>(pb, prm, b1, b2, b3, stream, two);
        case 160: return launch_bn<160, EPI_LINEAR>(pb, prm, b1, b2, b3, stream, two);
        case 128: return launch_bn<128, EPI_LINEAR>(pb, prm, b1, b2, b3, stream, two);
        case 64: return launch_bn<64, EPI_LINEAR>(pb, prm, b1, b2, b3, stream, two);
        default: break;
    }
    set_error("%s: unsupported tile width %d (256, 192, 160, 128, 64)", what, BN);
    return MVOC_ERR_UNSUPPORTED;
}

}  // namespace gemm
}  // namespace mvoc

using namespace mvoc;

extern "C" int mvoc_gemm_plan(int64_t rows, int64_t N, int geglu, int variant, int sms, int* tile_cols, int* cta_pair,
                              int* tail_cols) {
    MVOC_REQUIRE(tile_cols && cta_pair && tail_cols, MVOC_ERR_INVALID_ARG, "mvoc_gemm_plan: null pointer");
    MVOC_REQUIRE(rows > 0 && N > 0 && N % 64 == 0 && sms >= 2, MVOC_ERR_INVALID_ARG,
                 "mvoc_gemm_plan: rows=%lld N=%lld (a multiple of 64) sms=%d", (long long)rows, (long long)N, sms);
    int bn = 0;
    bool pair = false;
    gemm::plan_tiles((rows + gemm::BM - 1) / gemm::BM, N, geglu != 0, variant, sms, &bn, &pair);
    MVOC_REQUIRE(bn != 0, MVOC_ERR_UNSUPPORTED, "mvoc_gemm_plan: no tile width tiles N=%lld", (long long)N);
    *tile_cols = bn;
    *cta_pair = pair ? 1 : 0;
    *tail_cols = (int)(N % (geglu ? bn / 2 : bn));
    return MVOC_OK;
}

extern "C" int mvoc_conv3x3_nhwc(const void* x, const void* w_taps, const void* bias, const void* residual,
                                 const void* x2, const void* w2, int Cin2, void* out, int N, int H, int W, int Cin,
                                 int Cout, int dtype, int variant, void* stream) {
    gemm::Problem pb{};
    pb.what = "mvoc_conv3x3_nhwc";
    MVOC_REQUIRE(N > 0 && H > 0 && W > 0 && Cin > 0 && Cout > 0, MVOC_ERR_INVALID_ARG,
                 "%s: empty problem N=%d H=%d W=%d Cin=%d Cout=%d", pb.what, N, H, W, Cin, Cout);
    MVOC_REQUIRE((x2 == nullptr) == (w2 == nullptr), MVOC_ERR_INVALID_ARG, "%s: x2 and w2 go together", pb.what);
    pb.dtype = dtype;
    pb.d1 = W, pb.d2 = H, pb.d3 = N;
    pb.n_src = x2 ? 2 : 1;
    gemm::Source& s0 = pb.src[0];
    s0.a = x, s0.K = Cin, s0.w = w_taps, s0.taps = 9;
    s0.a_dim[0] = W, s0.a_dim[1] = H, s0.a_dim[2] = N, s0.stride = 1;
    s0.a_str[0] = Cin, s0.a_str[1] = (int64_t)W * Cin, s0.a_str[2] = (int64_t)H * W * Cin;
    for (int t = 0; t < 9; ++t) s0.off[t][0] = (int8_t)(t % 3 - 1), s0.off[t][1] = (int8_t)(t / 3 - 1), s0.off[t][2] = 0;
    if (x2) {
        gemm::Source& s1 = pb.src[1];
        s1.a = x2, s1.K = Cin2, s1.w = w2, s1.taps = 1;
        s1.a_dim[0] = W, s1.a_dim[1] = H, s1.a_dim[2] = N, s1.stride = 1;
        s1.a_str[0] = Cin2, s1.a_str[1] = (int64_t)W * Cin2, s1.a_str[2] = (int64_t)H * W * Cin2;
        s1.off[0][0] = s1.off[0][1] = s1.off[0][2] = 0;
    }
    pb.N = Cout, pb.w_rows = Cout;
    pb.bias = bias, pb.residual = residual, pb.out = out;
    pb.out_str[0] = Cout, pb.out_str[1] = (int64_t)W * Cout, pb.out_str[2] = (int64_t)H * W * Cout;
    for (int i = 0; i < 3; ++i) pb.res_str[i] = pb.out_str[i];
    pb.variant = variant;
    return gemm::run(pb, (cudaStream_t)stream);
}

extern "C" int mvoc_temporal_conv3(const void* x, const void* w_taps, const void* bias, const void* residual, void* out,
                                   int B, int T, int64_t S, int Cin, int Cout, int dtype, int variant, void* stream) {
    gemm::Problem pb{};
    pb.what = "mvoc_temporal_conv3";
    MVOC_REQUIRE(B > 0 && T > 0 && S > 0 && Cin > 0 && Cout > 0, MVOC_ERR_INVALID_ARG,
                 "%s: empty problem B=%d T=%d S=%lld Cin=%d Cout=%d", pb.what, B, T, (long long)S, Cin, Cout);
    pb.dtype = dtype;
    pb.d1 = S, pb.d2 = T, pb.d3 = B;
    pb.n_src = 1;
    gemm::Source& s0 = pb.src[0];
    s0.a = x, s0.K = Cin, s0.w = w_taps, s0.taps = 3;
    s0.a_dim[0] = S, s0.a_dim[1] = T, s0.a_dim[2] = B, s0.stride = 1;
    s0.a_str[0] = Cin, s0.a_str[1] = S * Cin, s0.a_str[2] = (int64_t)T * S * Cin;
    for (int t = 0; t < 3; ++t) s0.off[t][0] = 0, s0.off[t][1] = (int8_t)(t - 1), s0.off[t][2] = 0;
    pb.N = Cout, pb.w_rows = Cout;
    pb.bias = bias, pb.residual = residual, pb.out = out;
    pb.out_str[0] = Cout, pb.out_str[1] = S * Cout, pb.out_str[2] = (int64_t)T * S * Cout;
    for (int i = 0; i < 3; ++i) pb.res_str[i] = pb.out_str[i];
    pb.variant = variant;
    return gemm::run(pb, (cudaStream_t)stream);
}

extern "C" int mvoc_linear(const void* x, const void* w, const void* bias, const void* residual, void* out, int64_t M,
                           int K, int N, int64_t ldx, int64_t ldr, int64_t ldo, int dtype, int variant, void* stream) {
    gemm::Problem pb{};
    pb.what = "mvoc_linear";
    MVOC_REQUIRE(M > 0 && K > 0 && N > 0, MVOC_ERR_INVALID_ARG, "%s: empty problem M=%lld K=%d N=%d", pb.what,
                 (long long)M, K, N);
    MVOC_REQUIRE(ldx >= K && ldo >= N && (residual == nullptr || ldr >= N), MVOC_ERR_INVALID_ARG,
                 "%s: leading dimensions ldx=%lld ldr=%lld ldo=%lld too small for K=%d N=%d", pb.what, (long long)ldx,
                 (long long)ldr, (long long)ldo, K, N);
    pb.dtype = dtype;
    pb.d1 = M, pb.d2 = 1, pb.d3 = 1;
    pb.n_src = 1;
    gemm::Source& s0 = pb.src[0];
    s0.a = x, s0.K = K, s0.w = w, s0.taps = 1;
    s0.a_dim[0] = M, s0.a_dim[1] = 1, s0.a_dim[2] = 1, s0.stride = 1;
    s0.a_str[0] = ldx, s0.a_str[1] = 0, s0.a_str[2] = 0;
    s0.off[0][0] = s0.off[0][1] = s0.off[0][2] = 0;
    pb.N = N, pb.w_rows = N;
    pb.bias = bias, pb.residual = residual, pb.out = out;
    pb.out_str[0] = ldo, pb.out_str[1] = 0, pb.out_str[2] = 0;
    pb.res_str[0] = ldr, pb.res_str[1] = 0, pb.res_str[2] = 0;
    pb.variant = variant;
    return gemm::run(pb, (cudaStream_t)stream);
}

extern "C" int mvoc_linear_geglu(const void* x, const void* w, const void* bias, void* out, int64_t M, int K, int F,
                                 int dtype, int variant, void* stream) {
    gemm::Problem pb{};
    pb.what = "mvoc_linear_geglu";
    MVOC_REQUIRE(M > 0 && K > 0 && F > 0, MVOC_ERR_INVALID_ARG, "%s: empty problem M=%lld K=%d F=%d", pb.what,
                 (long long)M, K, F);
    pb.dtype = dtype;
    pb.d1 = M, pb.d2 = 1, pb.d3 = 1;
    pb.n_src = 1;
    gemm::Source& s0 = pb.src[0];
    s0.a = x, s0.K = K, s0.w = w, s0.taps = 1;
    s0.a_dim[0] = M, s0.a_dim[1] = 1, s0.a_dim[2] = 1, s0.stride = 1;
    s0.a_str[0] = K, s0.a_str[1] = 0, s0.a_str[2] = 0;
    s0.off[0][0] = s0.off[0][1] = s0.off[0][2] = 0;
    pb.N = F, pb.w_rows = 2 * (int64_t)F;
    pb.bias = bias, pb.residual = nullptr, pb.out = out;
    pb.out_str[0] = F, pb.out_str[1] = 0, pb.out_str[2] = 0;
    pb.geglu = 1;
    pb.variant = variant;
    return gemm::run(pb, (cudaStream_t)stream);
}

extern "C" int mvoc_conv3x3_s2_nhwc(const void* x, const void* w_taps, const void* bias, void* out, int N, int H, int W,
                                    int Cin, int Cout, int pad_begin, int pad_end, int dtype, int variant,
                                    void* stream) {
    gemm::Problem pb{};
    pb.what = "mvoc_conv3x3_s2_nhwc";
    MVOC_REQUIRE(N > 0 && H > 0 && W > 0 && Cin > 0 && Cout > 0, MVOC_ERR_INVALID_ARG,
                 "%s: empty problem N=%d H=%d W=%d Cin=%d Cout=%d", pb.what, N, H, W, Cin, Cout);
    MVOC_REQUIRE((pad_begin == 0 || pad_begin == 1) && (pad_end == 0 || pad_end == 1), MVOC_ERR_INVALID_ARG,
                 "%s: pad_begin=%d pad_end=%d (each 0 or 1)", pb.what, pad_begin, pad_end);
    // output extent of a 3-tap, stride-2 window over the padded axis (0 when the window does not fit once)
    auto out_extent = [&](int n) { return n + pad_begin + pad_end < 3 ? 0 : (n + pad_begin + pad_end - 3) / 2 + 1; };
    const int Ho = out_extent(H), Wo = out_extent(W);
    MVOC_REQUIRE(Ho >= 1 && Wo >= 1, MVOC_ERR_INVALID_ARG, "%s: H=%d W=%d with pads (%d, %d) leave an empty output",
                 pb.what, H, W, pad_begin, pad_end);
    pb.dtype = dtype;
    pb.d1 = Wo, pb.d2 = Ho, pb.d3 = N;
    pb.n_src = 1;
    gemm::Source& s0 = pb.src[0];
    s0.a = x, s0.K = Cin, s0.w = w_taps, s0.taps = 9;
    s0.a_dim[0] = W, s0.a_dim[1] = H, s0.a_dim[2] = N, s0.stride = 2;
    s0.a_str[0] = Cin, s0.a_str[1] = (int64_t)W * Cin, s0.a_str[2] = (int64_t)H * W * Cin;
    for (int t = 0; t < 9; ++t)
        s0.off[t][0] = (int8_t)(t % 3 - pad_begin), s0.off[t][1] = (int8_t)(t / 3 - pad_begin), s0.off[t][2] = 0;
    pb.N = Cout, pb.w_rows = Cout;
    pb.bias = bias, pb.residual = nullptr, pb.out = out;
    pb.out_str[0] = Cout, pb.out_str[1] = (int64_t)Wo * Cout, pb.out_str[2] = (int64_t)Ho * Wo * Cout;
    pb.variant = variant;
    return gemm::run(pb, (cudaStream_t)stream);
}

extern "C" int mvoc_linear_gelu(const void* x, const void* w, const void* bias, void* out, int64_t M, int K, int N,
                                int64_t ldx, int64_t ldo, int dtype, int variant, void* stream) {
    gemm::Problem pb{};
    pb.what = "mvoc_linear_gelu";
    MVOC_REQUIRE(M > 0 && K > 0 && N > 0, MVOC_ERR_INVALID_ARG, "%s: empty problem M=%lld K=%d N=%d", pb.what,
                 (long long)M, K, N);
    MVOC_REQUIRE(ldx >= K && ldo >= N, MVOC_ERR_INVALID_ARG, "%s: leading dimensions ldx=%lld ldo=%lld too small for K=%d N=%d",
                 pb.what, (long long)ldx, (long long)ldo, K, N);
    pb.dtype = dtype;
    pb.d1 = M, pb.d2 = 1, pb.d3 = 1;
    pb.n_src = 1;
    gemm::Source& s0 = pb.src[0];
    s0.a = x, s0.K = K, s0.w = w, s0.taps = 1;
    s0.a_dim[0] = M, s0.a_dim[1] = 1, s0.a_dim[2] = 1, s0.stride = 1;
    s0.a_str[0] = ldx, s0.a_str[1] = 0, s0.a_str[2] = 0;
    s0.off[0][0] = s0.off[0][1] = s0.off[0][2] = 0;
    pb.N = N, pb.w_rows = N;
    pb.bias = bias, pb.residual = nullptr, pb.out = out;
    pb.out_str[0] = ldo, pb.out_str[1] = 0, pb.out_str[2] = 0;
    pb.gelu = 1;
    pb.variant = variant;
    return gemm::run(pb, (cudaStream_t)stream);
}
