// Tensor-core attention forward for ONE head of width 512 on sm_100a (tcgen05 + TMEM + TMA).
// Reference: the mid-block Attention of diffusers' AutoencoderKL decoder (single head, head_dim = 512 channels),
// reached from decode_latents, i2vgen-xl/pipelines/pipeline_i2vgen_xl.py:771-791.  Non-causal, no mask.
//
// Budget at D = 512: the O accumulator of a 128-row tile is 512 fp32 TMEM columns (all of TMEM) and the Q tile is
// 128 KB of shared memory.  So the value dimension is split over two CTAs per Q tile (blockIdx.y = half): each
// recomputes S = Q K^T over the full 512 and owns 256 O columns.  1.5x the MMA work of an ideal kernel, but every
// accumulator fits one CTA: TMEM columns S [0,128)  P [128,192) (16-bit pairs)  O [256,512).
//
// One CTA = one 128-row query tile x one half of the value columns; one CTA per SM (224 KB of shared memory).
//   warps 0-3  softmax: thread i owns query row i (= TMEM lane i); the 128-key score row lives in registers
//   warp  4    TMA producer: Q once (8 boxes of 128 rows x 64), then a ring of 32 KB slots
//   warp  5    MMA issuer (one lane); owns the TMEM allocation
// Slot stream, in the order the MMA lane consumes it: K(0) as 4 slots of 128 keys x 128 dims, then per key block j
// the 4 K slots of block j+1 followed by the 2 V slots of block j (128 keys x 128 of this CTA's value columns).
// Q, K, V are read through 4-D tensor maps that view a row of 512 as 8 boxes of 64 (128-byte swizzle), so the
// three column slices of a fused QKV projection output are read in place.  Ragged N: TMA zero-fills rows past N,
// the scores of those keys are set to -inf, and rows past N are not stored.
#include <cuda.h>
#include <type_traits>
#include "common.cuh"
#include "ptx.cuh"

namespace mvoc {
namespace attn_wide {

constexpr int BM = 128;             // query rows per CTA
constexpr int BN = 128;             // keys per block
constexpr int D = 512;              // head dim
constexpr int DV = D / 2;           // value columns per CTA
constexpr int BOX = 64;             // 16-bit elements per 128-byte swizzle row
constexpr int BOX_BYTES = 128 * BOX * 2;     // 16 KB: 128 rows x 128 B
constexpr int SLOT_BYTES = 2 * BOX_BYTES;    // 32 KB: 128 rows x 128 columns
constexpr int STAGES = 3;
constexpr int K_SLOTS = D / 128;    // 4 slots per K block
constexpr int V_SLOTS = DV / 128;   // 2 slots per V block
constexpr int THREADS = 192;
constexpr uint32_t TMEM_COLS = 512;
constexpr uint32_t COL_S = 0, COL_P = 128, COL_O = 256;
constexpr float RESCALE_LOG2_THRESHOLD = 8.0f;

constexpr int Q_OFF = 0;
constexpr int RING_OFF = Q_OFF + (D / BOX) * BOX_BYTES;
constexpr int BAR_OFF = RING_OFF + STAGES * SLOT_BYTES;
// barriers: q_full, s_full, s_free, p_full, pv_done, slot_full[STAGES], slot_empty[STAGES]
constexpr int N_BARS = 5 + 2 * STAGES;
constexpr int TMEM_PTR_OFF = BAR_OFF + N_BARS * 8;
constexpr int SMEM_BYTES = TMEM_PTR_OFF + 16;
static_assert(SMEM_BYTES + 1024 <= 233472, "the CTA no longer fits the shared memory of an SM");
static_assert(COL_O + DV <= TMEM_COLS, "S + P + O exceed the TMEM columns");

struct Params {
    void* o;
    int64_t o_sb, o_sn;
    int N;
    float scale_log2;
};

template <typename T>
__global__ void __launch_bounds__(THREADS, 1)
attn_d512_kernel(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_k,
                 const __grid_constant__ CUtensorMap tm_v, const Params prm) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const uint32_t sbase = smem_u32(smem_raw);
    MVOC_REQUIRE_SMEM_1024(sbase, "attn_d512_kernel");
    const uint32_t sQ = sbase + Q_OFF;
    const uint32_t sRing = sbase + RING_OFF;
    const uint32_t bars = sbase + BAR_OFF;
    const uint32_t b_q_full = bars, b_s_full = bars + 8, b_s_free = bars + 16, b_p_full = bars + 24,
                   b_pv_done = bars + 32;
    const uint32_t b_slot_full = bars + 40, b_slot_empty = b_slot_full + 8 * STAGES;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m_blk = blockIdx.x, half = blockIdx.y, b = blockIdx.z;
    const int n_blocks = (prm.N + BN - 1) / BN;

    if (warp == 4 && lane == 0) {
        ptx::prefetch_tensormap(&tm_q);
        ptx::prefetch_tensormap(&tm_k);
        ptx::prefetch_tensormap(&tm_v);
        ptx::mbar_init(b_q_full, 1);
        ptx::mbar_init(b_s_full, 1);
        ptx::mbar_init(b_s_free, 4);     // one arrival per softmax warp
        ptx::mbar_init(b_p_full, 4);
        ptx::mbar_init(b_pv_done, 1);
        for (int s = 0; s < STAGES; ++s) {
            ptx::mbar_init(b_slot_full + 8 * s, 1);
            ptx::mbar_init(b_slot_empty + 8 * s, 1);
        }
        ptx::fence_mbar_init();
    }
    if (warp == 5) {
        ptx::tmem_alloc(sbase + TMEM_PTR_OFF, TMEM_COLS);
        ptx::tmem_relinquish();
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(smem_raw + TMEM_PTR_OFF);

    if (warp == 4) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            ptx::mbar_expect_tx(b_q_full, (D / BOX) * BOX_BYTES);
            for (int c = 0; c < D / BOX; ++c)
                ptx::tma_load_4d(sQ + c * BOX_BYTES, &tm_q, b_q_full, 0, c, m_blk * BM, b);
        }
        int u = 0;  // slot-stream position
        // box index (of 8 along the 512 columns) pair `first`, `first + 1` of key block j into the next slot
        auto load_slot = [&](const CUtensorMap* tm, int first, int j) {
            const int s = u % STAGES;
            ptx::mbar_wait(b_slot_empty + 8 * s, ((uint32_t)(u / STAGES) & 1u) ^ 1u, 20);
            if (lane == 0) {
                const uint32_t dst = sRing + s * SLOT_BYTES;
                ptx::mbar_expect_tx(b_slot_full + 8 * s, SLOT_BYTES);
                ptx::tma_load_4d(dst, tm, b_slot_full + 8 * s, 0, first, j * BN, b);
                ptx::tma_load_4d(dst + BOX_BYTES, tm, b_slot_full + 8 * s, 0, first + 1, j * BN, b);
            }
            __syncwarp();
            ++u;
        };
        for (int c = 0; c < K_SLOTS; ++c) load_slot(&tm_k, 2 * c, 0);
        for (int j = 0; j < n_blocks; ++j) {
            if (j + 1 < n_blocks)
                for (int c = 0; c < K_SLOTS; ++c) load_slot(&tm_k, 2 * c, j + 1);
            for (int c = 0; c < V_SLOTS; ++c) load_slot(&tm_v, half * (DV / BOX) + 2 * c, j);
        }
    } else if (warp == 5) {
        // ===================== MMA issuer =====================
        constexpr bool kF16 = std::is_same<T, __half>::value;
        constexpr uint32_t IDESC_QK = ptx::idesc_f16(kF16, BM, BN, false);  // A (Q), B (K) K-major
        constexpr uint32_t IDESC_PV = ptx::idesc_f16(kF16, BM, BOX, true);  // B (V) MN-major, 64 value columns per MMA
        const uint32_t tS = tmem + COL_S, tP = tmem + COL_P, tO = tmem + COL_O;
        int u = 0;
        auto wait_slot = [&]() {
            const int s = u % STAGES;
            ptx::mbar_wait(b_slot_full + 8 * s, (uint32_t)(u / STAGES) & 1u, 21);
            ptx::tc_fence_after();
            return s;
        };
        auto issue_qk = [&]() {
            for (int c = 0; c < K_SLOTS; ++c) {
                const int s = wait_slot();
                if (lane == 0) {
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const uint64_t a0 = ptx::smem_desc_sw128(sQ + (2 * c + e) * BOX_BYTES, 16, 1024);
                        const uint64_t b0 = ptx::smem_desc_sw128(sRing + s * SLOT_BYTES + e * BOX_BYTES, 16, 1024);
#pragma unroll
                        for (int ks = 0; ks < BOX / 16; ++ks)  // +32 B per 16-element K step (encoded >>4)
                            ptx::mma_ss(tS, a0 + (uint64_t)(ks * 2), b0 + (uint64_t)(ks * 2), IDESC_QK,
                                        (c > 0 || e > 0 || ks > 0) ? 1u : 0u);
                    }
                    ptx::tc_commit(b_slot_empty + 8 * s);
                }
                __syncwarp();
                ++u;
            }
            if (lane == 0) ptx::tc_commit(b_s_full);
            __syncwarp();
        };
        ptx::mbar_wait(b_q_full, 0, 22);
        ptx::tc_fence_after();
        issue_qk();
        for (int j = 0; j < n_blocks; ++j) {
            if (j + 1 < n_blocks) {
                ptx::mbar_wait(b_s_free, (uint32_t)j & 1u, 23);   // S of block j sits in registers
                ptx::tc_fence_after();
                issue_qk();
            }
            ptx::mbar_wait(b_p_full, (uint32_t)j & 1u, 24);
            ptx::tc_fence_after();
            for (int c = 0; c < V_SLOTS; ++c) {
                const int s = wait_slot();
                if (lane == 0) {
                    // V box: rows = keys (K of this GEMM), 128 B per row = 64 value columns (N) contiguous
#pragma unroll
                    for (int g = 0; g < 2; ++g) {
                        const uint64_t bv = ptx::smem_desc_sw128(sRing + s * SLOT_BYTES + g * BOX_BYTES, 16384, 1024);
#pragma unroll
                        for (int ks = 0; ks < BN / 16; ++ks)
                            ptx::mma_ts(tO + (2 * c + g) * BOX, tP + ks * 8, bv + (uint64_t)((ks * 2048) >> 4),
                                        IDESC_PV, (j > 0 || ks > 0) ? 1u : 0u);
                    }
                    ptx::tc_commit(b_slot_empty + 8 * s);
                }
                __syncwarp();
                ++u;
            }
            if (lane == 0) ptx::tc_commit(b_pv_done);
            __syncwarp();
        }
    } else {
        // ===================== softmax + epilogue (warps 0-3) =====================
        const int row = threadIdx.x;  // query row inside the tile == TMEM lane
        const uint32_t lane_base = tmem + ((uint32_t)(warp * 32) << 16);
        const uint32_t tS = lane_base + COL_S, tP = lane_base + COL_P, tO = lane_base + COL_O;
        const float sl2 = prm.scale_log2;
        float m_used = -INFINITY, l_sum = 0.0f;
        for (int j = 0; j < n_blocks; ++j) {
            const int valid = min(BN, prm.N - j * BN);
            ptx::mbar_wait(b_s_full, (uint32_t)j & 1u, 25);
            ptx::tc_fence_after();
            uint32_t r[BN];
#pragma unroll
            for (int c = 0; c < BN / 32; ++c)
                ptx::tmem_ld32(tS + c * 32, *reinterpret_cast<uint32_t(*)[32]>(&r[c * 32]));
            ptx::tmem_wait_ld();
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(b_s_free);
            if (valid < BN) {  // keys past N (zero-filled by TMA) must not take part: exp2(-inf) = 0
#pragma unroll
                for (int i = 0; i < BN; ++i)
                    if (i >= valid) r[i] = 0xff800000u;
            }
            float mxc[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) mxc[e] = -INFINITY;
#pragma unroll
            for (int i = 0; i < BN; i += 16) {
#pragma unroll
                for (int e = 0; e < 8; ++e)
                    mxc[e] = ptx::max3(mxc[e], __uint_as_float(r[i + 2 * e]), __uint_as_float(r[i + 2 * e + 1]));
            }
            const float mx = fmaxf(ptx::max3(mxc[0], mxc[1], mxc[2]),
                                   fmaxf(ptx::max3(mxc[3], mxc[4], mxc[5]), fmaxf(mxc[6], mxc[7])));
            bool pv_waited = (j == 0);   // the previous P V is known complete
            if (j == 0) {
                m_used = mx;
            } else {
                const float m_new = fmaxf(m_used, mx);
                const bool need = (m_new - m_used) * sl2 > RESCALE_LOG2_THRESHOLD;
                if (__any_sync(0xffffffffu, need)) {
                    // rescale the running O and l (rare after the first blocks)
                    ptx::mbar_wait(b_pv_done, (uint32_t)(j - 1) & 1u, 26);
                    ptx::tc_fence_after();
                    pv_waited = true;
                    const float f = need ? ptx::ex2_approx((m_used - m_new) * sl2) : 1.0f;
                    if (need) m_used = m_new;
                    l_sum *= f;
#pragma unroll 1
                    for (int c = 0; c < DV / 32; ++c) {
                        uint32_t o[32];
                        ptx::tmem_ld32(tO + c * 32, o);
                        ptx::tmem_wait_ld();
#pragma unroll
                        for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * f);
                        ptx::tmem_st32(tO + c * 32, o);
                    }
                    ptx::tmem_wait_st();
                }
            }
            // p = exp2(s * scale*log2e - m * scale*log2e) on pairs (FFMA2), packed row sums (FADD2)
            const uint64_t sl2_2 = ptx::pack2(sl2, sl2);
            const uint64_t negm_2 = ptx::pack2(-m_used * sl2, -m_used * sl2);
            uint32_t pk[BN / 2];
            uint64_t la = ptx::pack2(0.0f, 0.0f), lb = la;
#pragma unroll
            for (int k = 0; k < BN / 2; ++k) {
                const uint64_t x2 = ptx::fma2(ptx::pack2(__uint_as_float(r[2 * k]), __uint_as_float(r[2 * k + 1])),
                                              sl2_2, negm_2);
                float x0, x1;
                ptx::unpack2(x2, x0, x1);
                const float p0 = ptx::ex2_approx(x0), p1 = ptx::ex2_approx(x1);
                if (k & 1) lb = ptx::add2(lb, ptx::pack2(p0, p1));
                else la = ptx::add2(la, ptx::pack2(p0, p1));
                pk[k] = pack2_rn<T>(p0, p1);
            }
            {
                float s0, s1;
                ptx::unpack2(ptx::add2(la, lb), s0, s1);
                l_sum += s0 + s1;
            }
            // the P buffer is free once the previous P V has completed
            if (!pv_waited) {
                ptx::mbar_wait(b_pv_done, (uint32_t)(j - 1) & 1u, 27);
                ptx::tc_fence_after();
            }
#pragma unroll
            for (int c = 0; c < BN / 64; ++c)
                ptx::tmem_st32(tP + c * 32, *reinterpret_cast<uint32_t(*)[32]>(&pk[c * 32]));
            ptx::tmem_wait_st();
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(b_p_full);
        }
        // ---- epilogue: O / l -> 16-bit -> global --------------------------------
        ptx::mbar_wait(b_pv_done, (uint32_t)(n_blocks - 1) & 1u, 28);
        ptx::tc_fence_after();
        const float inv_l = 1.0f / l_sum;
        const int q_row = m_blk * BM + row;
        T* orow = reinterpret_cast<T*>(prm.o) + (int64_t)b * prm.o_sb + (int64_t)q_row * prm.o_sn + half * DV;
#pragma unroll 1
        for (int c = 0; c < DV / 32; ++c) {
            uint32_t r[32];
            ptx::tmem_ld32(tO + c * 32, r);
            ptx::tmem_wait_ld();
            if (q_row < prm.N) {
#pragma unroll
                for (int i = 0; i < 32; i += 8) {
                    float f[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) f[e] = __uint_as_float(r[i + e]) * inv_l;
                    *reinterpret_cast<Vec16*>(orow + c * 32 + i) = pack8<T>(f);
                }
            }
        }
        ptx::tc_fence_before();
    }

    __syncthreads();
    if (warp == 5) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc(tmem, TMEM_COLS);
    }
}

// ------------------------------------------------------------------ host ---
template <typename T>
static int launch(const CUtensorMap (&m)[3], const Params& prm, int B, cudaStream_t s, const char* what) {
    static bool smem_set[64] = {false};
    const int rc = set_max_dynamic_smem((const void*)attn_d512_kernel<T>, SMEM_BYTES, smem_set, what);
    if (rc != MVOC_OK) return rc;
    dim3 grid((prm.N + BM - 1) / BM, 2, B);
    attn_d512_kernel<T><<<grid, THREADS, SMEM_BYTES, s>>>(m[0], m[1], m[2], prm);
    return check_launch(what);
}

}  // namespace attn_wide
}  // namespace mvoc

using namespace mvoc;

extern "C" int mvoc_attn_d512_fwd(const void* q, const void* k, const void* v, void* o, int B, int N, int D,
                                  int64_t q_sb, int64_t q_sn, int64_t k_sb, int64_t k_sn, int64_t v_sb,
                                  int64_t v_sn, int64_t o_sb, int64_t o_sn, float scale, int dtype, void* stream) {
    using namespace attn_wide;
    const char* what = "mvoc_attn_d512_fwd";
    const int64_t st[8] = {q_sb, q_sn, k_sb, k_sn, v_sb, v_sn, o_sb, o_sn};
    int rc = check_attn_operands(q, k, v, o, dtype, D, attn_wide::D, st, 8, what);
    if (rc != MVOC_OK) return rc;
    MVOC_REQUIRE(B > 0 && N > 0, MVOC_ERR_INVALID_ARG, "%s: empty problem B=%d N=%d", what, B, N);
    MVOC_REQUIRE(B <= 65535, MVOC_ERR_UNSUPPORTED, "%s: B=%d exceeds the grid limit", what, B);
    // q, k, v: [B, N, 512] viewed innermost first as [64, 8, N, B]; box = 64 columns of 128 tokens
    const void* ptr[3] = {q, k, v};
    const char* name[3] = {"q", "k", "v"};
    const int64_t dims[4] = {BOX, attn_wide::D / BOX, N, B};
    const int64_t str[3][3] = {{BOX, q_sn, q_sb}, {BOX, k_sn, k_sb}, {BOX, v_sn, v_sb}};
    const int box[4] = {BOX, 1, BM, 1};
    for (int i = 0; i < 3; ++i)   // all three before the first driver call
        if ((rc = check_map4(dims, str[i], what, name[i])) != MVOC_OK) return rc;
    CUtensorMap m[3];
    for (int i = 0; i < 3; ++i)
        if ((rc = make_map4(&m[i], ptr[i], dtype, dims, str[i], box, 1, CU_TENSOR_MAP_SWIZZLE_128B, what, name[i])) !=
            MVOC_OK)
            return rc;
    Params prm;
    prm.o = o;
    prm.o_sb = o_sb;
    prm.o_sn = o_sn;
    prm.N = N;
    prm.scale_log2 = scale * 1.4426950408889634f;
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == MVOC_F16) return launch<__half>(m, prm, B, s, what);
    return launch<__nv_bfloat16>(m, prm, B, s, what);
}
