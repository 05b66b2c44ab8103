// Tensor-core attention forward at head_dim 80 on sm_100a (tcgen05 + TMEM + TMA).
// Reference: the self-attention of transformers' CLIPAttention in the CLIP image tower (CLIPVisionModelWithProjection,
// ViT-H/14: 16 heads of 80 over 257 tokens), called from I2VGenXLPipeline._encode_image, pipeline_i2vgen_xl.py:
// 1391-1541 of the reference.  Non-causal, no mask, no dropout.
//
// An 80-element 16-bit row is 160 bytes, wider than the 128-byte swizzle span.  Each operand tile is therefore TWO
// 128-byte-swizzled boxes of 64 columns: columns [0, 64) and [64, 128), where the tensor map's innermost extent of 80
// makes TMA zero-fill columns [80, 128) (the next head's columns are never read).  80 = 5 x 16:
//   S = Q K^T    four K = 16 steps in box 0 and one in box 1 (the zero-filled columns are not multiplied)
//   O += P V     one N = 80 MMA per 16 keys: V is MN-major, its 64-column swizzle atoms 16 KB (one box) apart (LBO)
// TMEM columns (fp32): S [0,128)  P [128,192) (16-bit pairs)  O [256,336); the allocation is 512 (one CTA per SM).
//
// One CTA = one 128-row query tile of one (batch, head).
//   warps 0-3  softmax: thread i owns query row i (= TMEM lane i); the 128-key score row lives in registers
//   warp  4    TMA producer: Q once, then a ring of 32 KB slots (one K or V block of 128 keys each)
//   warp  5    MMA issuer (one lane); owns the TMEM allocation
// Slot stream, in the order the MMA lane consumes it: K(0), then per key block j: K(j+1), V(j).
// Ragged N: TMA zero-fills rows past N, the scores of those keys are set to -inf, and rows past N are not stored.
#include <cuda.h>
#include <type_traits>
#include "common.cuh"
#include "ptx.cuh"

namespace mvoc {
namespace attn_d80 {

constexpr int BM = 128;             // query rows per CTA
constexpr int BN = 128;             // keys per block
constexpr int D = 80;               // head dim
constexpr int BOX = 64;             // 16-bit elements per 128-byte swizzle row
constexpr int BOX_BYTES = 128 * BOX * 2;     // 16 KB: 128 rows x 128 B
constexpr int SLOT_BYTES = 2 * BOX_BYTES;    // 32 KB: 128 rows x 128 columns (80 real + 48 zero-filled)
constexpr int STAGES = 4;
constexpr int THREADS = 192;
constexpr uint32_t TMEM_COLS = 512;
constexpr uint32_t COL_S = 0, COL_P = 128, COL_O = 256;
constexpr float RESCALE_LOG2_THRESHOLD = 8.0f;

constexpr int Q_OFF = 0;
constexpr int RING_OFF = Q_OFF + SLOT_BYTES;
constexpr int BAR_OFF = RING_OFF + STAGES * SLOT_BYTES;
// barriers: q_full, s_full, s_free, p_full, pv_done, slot_full[STAGES], slot_empty[STAGES]
constexpr int N_BARS = 5 + 2 * STAGES;
constexpr int TMEM_PTR_OFF = BAR_OFF + N_BARS * 8;
constexpr int SMEM_BYTES = TMEM_PTR_OFF + 16;
static_assert(SMEM_BYTES + 1024 <= 233472, "the CTA no longer fits the shared memory of an SM");
static_assert(COL_O + 96 <= TMEM_COLS, "S + P + O (read in 32-column pieces) exceed the TMEM columns");
static_assert(D % 16 == 0 && D > BOX && D <= 2 * BOX, "head dim: two boxes, whole K = 16 steps");

struct Params {
    void* o;
    int64_t o_sb, o_sn, o_sh;
    int Nq, Nk;
    float scale_log2;
};

template <typename T>
__global__ void __launch_bounds__(THREADS, 1)
attn_d80_kernel(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_k,
                const __grid_constant__ CUtensorMap tm_v, const Params prm) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const uint32_t sbase = smem_u32(smem_raw);
    MVOC_REQUIRE_SMEM_1024(sbase, "attn_d80_kernel");
    const uint32_t sQ = sbase + Q_OFF;
    const uint32_t sRing = sbase + RING_OFF;
    const uint32_t bars = sbase + BAR_OFF;
    const uint32_t b_q_full = bars, b_s_full = bars + 8, b_s_free = bars + 16, b_p_full = bars + 24,
                   b_pv_done = bars + 32;
    const uint32_t b_slot_full = bars + 40, b_slot_empty = b_slot_full + 8 * STAGES;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m_blk = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
    const int n_blocks = (prm.Nk + BN - 1) / BN;

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
            ptx::mbar_expect_tx(b_q_full, SLOT_BYTES);
            ptx::tma_load_4d(sQ, &tm_q, b_q_full, 0, h, m_blk * BM, b);
            ptx::tma_load_4d(sQ + BOX_BYTES, &tm_q, b_q_full, BOX, h, m_blk * BM, b);
        }
        int u = 0;  // slot-stream position
        auto load_slot = [&](const CUtensorMap* tm, int j) {   // key block j of K or V: both boxes
            const int s = u % STAGES;
            ptx::mbar_wait(b_slot_empty + 8 * s, ((uint32_t)(u / STAGES) & 1u) ^ 1u, 40);
            if (lane == 0) {
                const uint32_t dst = sRing + s * SLOT_BYTES;
                ptx::mbar_expect_tx(b_slot_full + 8 * s, SLOT_BYTES);
                ptx::tma_load_4d(dst, tm, b_slot_full + 8 * s, 0, h, j * BN, b);
                ptx::tma_load_4d(dst + BOX_BYTES, tm, b_slot_full + 8 * s, BOX, h, j * BN, b);
            }
            __syncwarp();
            ++u;
        };
        load_slot(&tm_k, 0);
        for (int j = 0; j < n_blocks; ++j) {
            if (j + 1 < n_blocks) load_slot(&tm_k, j + 1);
            load_slot(&tm_v, j);
        }
    } else if (warp == 5) {
        // ===================== MMA issuer =====================
        constexpr bool kF16 = std::is_same<T, __half>::value;
        constexpr uint32_t IDESC_QK = ptx::idesc_f16(kF16, BM, BN, false);  // A (Q), B (K) K-major
        constexpr uint32_t IDESC_PV = ptx::idesc_f16(kF16, BM, D, true);    // B (V) MN-major, all 80 value columns
        const uint32_t tS = tmem + COL_S, tP = tmem + COL_P, tO = tmem + COL_O;
        int u = 0;
        auto wait_slot = [&]() {
            const int s = u % STAGES;
            ptx::mbar_wait(b_slot_full + 8 * s, (uint32_t)(u / STAGES) & 1u, 41);
            ptx::tc_fence_after();
            return s;
        };
        auto issue_qk = [&]() {
            const int s = wait_slot();
            if (lane == 0) {
#pragma unroll
                for (int ks = 0; ks < D / 16; ++ks) {   // +32 B per 16-element K step (encoded >>4) inside a box
                    const int e = ks / 4, kb = ks % 4;
                    const uint64_t a = ptx::smem_desc_sw128(sQ + e * BOX_BYTES, 16, 1024) + (uint64_t)(kb * 2);
                    const uint64_t bk =
                        ptx::smem_desc_sw128(sRing + s * SLOT_BYTES + e * BOX_BYTES, 16, 1024) + (uint64_t)(kb * 2);
                    ptx::mma_ss(tS, a, bk, IDESC_QK, ks > 0 ? 1u : 0u);
                }
                ptx::tc_commit(b_slot_empty + 8 * s);
                ptx::tc_commit(b_s_full);
            }
            __syncwarp();
            ++u;
        };
        ptx::mbar_wait(b_q_full, 0, 42);
        ptx::tc_fence_after();
        issue_qk();
        for (int j = 0; j < n_blocks; ++j) {
            if (j + 1 < n_blocks) {
                ptx::mbar_wait(b_s_free, (uint32_t)j & 1u, 43);   // S of block j sits in registers
                ptx::tc_fence_after();
                issue_qk();
            }
            ptx::mbar_wait(b_p_full, (uint32_t)j & 1u, 44);
            ptx::tc_fence_after();
            const int s = wait_slot();
            if (lane == 0) {
                // V slot: rows = keys (K of this GEMM), 128 B per row and box = 64 value columns (N) contiguous;
                // value columns 64..79 are the first 32 B of the rows of box 1, one LBO further
                const uint64_t bv = ptx::smem_desc_sw128(sRing + s * SLOT_BYTES, BOX_BYTES, 1024);
#pragma unroll
                for (int ks = 0; ks < BN / 16; ++ks)
                    ptx::mma_ts(tO, tP + ks * 8, bv + (uint64_t)((ks * 2048) >> 4), IDESC_PV, (j > 0 || ks > 0) ? 1u : 0u);
                ptx::tc_commit(b_slot_empty + 8 * s);
                ptx::tc_commit(b_pv_done);
            }
            __syncwarp();
            ++u;
        }
    } else {
        // ===================== softmax + epilogue (warps 0-3) =====================
        const int row = threadIdx.x;  // query row inside the tile == TMEM lane
        const uint32_t lane_base = tmem + ((uint32_t)(warp * 32) << 16);
        const uint32_t tS = lane_base + COL_S, tP = lane_base + COL_P, tO = lane_base + COL_O;
        const float sl2 = prm.scale_log2;
        float m_used = -INFINITY, l_sum = 0.0f;
        for (int j = 0; j < n_blocks; ++j) {
            const int valid = min(BN, prm.Nk - j * BN);
            ptx::mbar_wait(b_s_full, (uint32_t)j & 1u, 45);
            ptx::tc_fence_after();
            uint32_t r[BN];
#pragma unroll
            for (int c = 0; c < BN / 32; ++c)
                ptx::tmem_ld32(tS + c * 32, *reinterpret_cast<uint32_t(*)[32]>(&r[c * 32]));
            ptx::tmem_wait_ld();
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(b_s_free);
            if (valid < BN) {  // keys past Nk (zero-filled by TMA) must not take part: exp2(-inf) = 0
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
                    // rescale the running O and l (rare after the first blocks); the third piece carries 16 unused
                    // columns along
                    ptx::mbar_wait(b_pv_done, (uint32_t)(j - 1) & 1u, 46);
                    ptx::tc_fence_after();
                    pv_waited = true;
                    const float f = need ? ptx::ex2_approx((m_used - m_new) * sl2) : 1.0f;
                    if (need) m_used = m_new;
                    l_sum *= f;
#pragma unroll 1
                    for (int c = 0; c < (D + 31) / 32; ++c) {
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
                ptx::mbar_wait(b_pv_done, (uint32_t)(j - 1) & 1u, 47);
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
        ptx::mbar_wait(b_pv_done, (uint32_t)(n_blocks - 1) & 1u, 48);
        ptx::tc_fence_after();
        const float inv_l = 1.0f / l_sum;
        const int q_row = m_blk * BM + row;
        T* orow = reinterpret_cast<T*>(prm.o) + (int64_t)b * prm.o_sb + (int64_t)q_row * prm.o_sn +
                  (int64_t)h * prm.o_sh;
#pragma unroll
        for (int c = 0; c < (D + 31) / 32; ++c) {
            uint32_t r[32];
            ptx::tmem_ld32(tO + c * 32, r);
            ptx::tmem_wait_ld();
            if (q_row < prm.Nq) {
#pragma unroll
                for (int i = 0; i < 32; i += 8) {
                    if (c * 32 + i >= D) break;
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
static int launch(const CUtensorMap (&m)[3], const Params& prm, int B, int H, cudaStream_t s, const char* what) {
    static bool smem_set[64] = {false};
    const int rc = set_max_dynamic_smem((const void*)attn_d80_kernel<T>, SMEM_BYTES, smem_set, what);
    if (rc != MVOC_OK) return rc;
    dim3 grid((prm.Nq + BM - 1) / BM, H, B);
    attn_d80_kernel<T><<<grid, THREADS, SMEM_BYTES, s>>>(m[0], m[1], m[2], prm);
    return check_launch(what);
}

}  // namespace attn_d80
}  // namespace mvoc

using namespace mvoc;

extern "C" int mvoc_attn_d80_fwd(const void* q, const void* k, const void* v, void* o, int B, int H, int Nq, int Nk,
                                 int D, int64_t q_sb, int64_t q_sn, int64_t q_sh, int64_t k_sb, int64_t k_sn,
                                 int64_t k_sh, int64_t v_sb, int64_t v_sn, int64_t v_sh, int64_t o_sb, int64_t o_sn,
                                 int64_t o_sh, float scale, int dtype, void* stream) {
    using namespace attn_d80;
    const char* what = "mvoc_attn_d80_fwd";
    const int64_t st[12] = {q_sb, q_sn, q_sh, k_sb, k_sn, k_sh, v_sb, v_sn, v_sh, o_sb, o_sn, o_sh};
    int rc = check_attn_operands(q, k, v, o, dtype, D, attn_d80::D, st, 12, what);
    if (rc != MVOC_OK) return rc;
    MVOC_REQUIRE(B > 0 && H > 0 && Nq > 0 && Nk > 0, MVOC_ERR_INVALID_ARG, "%s: empty problem B=%d H=%d Nq=%d Nk=%d",
                 what, B, H, Nq, Nk);
    MVOC_REQUIRE(B <= 65535 && H <= 65535, MVOC_ERR_UNSUPPORTED, "%s: B=%d / H=%d exceed the grid limits", what, B, H);
    // q, k, v: [B, N, H, 80] viewed innermost first with element strides (sh, sn, sb); box = 64 columns of 128 tokens,
    // taken at columns 0 and 64 (the second box zero-filled past column 80)
    const void* ptr[3] = {q, k, v};
    const char* name[3] = {"q", "k", "v"};
    const int64_t dims[3][4] = {{attn_d80::D, H, Nq, B}, {attn_d80::D, H, Nk, B}, {attn_d80::D, H, Nk, B}};
    const int64_t str[3][3] = {{q_sh, q_sn, q_sb}, {k_sh, k_sn, k_sb}, {v_sh, v_sn, v_sb}};
    const int box[4] = {BOX, 1, BM, 1};
    for (int i = 0; i < 3; ++i)   // all three before the first driver call
        if ((rc = check_map4(dims[i], str[i], what, name[i])) != MVOC_OK) return rc;
    CUtensorMap m[3];
    for (int i = 0; i < 3; ++i)
        if ((rc = make_map4(&m[i], ptr[i], dtype, dims[i], str[i], box, 1, CU_TENSOR_MAP_SWIZZLE_128B, what,
                            name[i])) != MVOC_OK)
            return rc;
    Params prm;
    prm.o = o;
    prm.o_sb = o_sb;
    prm.o_sn = o_sn;
    prm.o_sh = o_sh;
    prm.Nq = Nq;
    prm.Nk = Nk;
    prm.scale_log2 = scale * 1.4426950408889634f;
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == MVOC_F16) return launch<__half>(m, prm, B, H, s, what);
    return launch<__nv_bfloat16>(m, prm, B, H, s, what);
}
