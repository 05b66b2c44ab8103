// Tensor-core flash attention forward for sm_100a (tcgen05 + TMEM + TMA).
// Reference: F.scaled_dot_product_attention at i2vgen-xl/pnp_utils.py:684-686
// and inside diffusers' AttnProcessor2_0 (reached through attention_forward,
// i2vgen-xl/pnp_utils.py:348-385) — non-causal, no mask, no dropout, D = 64.
//
// Causal mode (kCausal, mvoc_attn_causal_fwd; the CLIP text tower's self-attention): Nq == Nk, query row r sees keys
// 0..r.  Query tile m needs key blocks 0..m only (BM == BN), so the producer, MMA and softmax warps all run
// min(ceil(Nk/128), m + 1) blocks: blocks above the diagonal are never loaded, multiplied or exponentiated.  In the
// diagonal block, columns past the row are set to -inf by the same register select as the tail mask.
//
// Pair mode (kNV = 2): MVOC writes the SAME blended Q', K' to the uncond and cond composite slots
// (i2vgen-xl/pnp_utils.py:664-668), so their score matrices are identical: one CTA computes S and the softmax once
// and multiplies P with BOTH value tiles (two O accumulators) — half the exponentials for those two branches.  It
// runs on 64-key blocks so that S + P + 2 O still fit the 256 TMEM columns that let two CTAs share an SM.
// bf16 or fp16 storage (P is rounded to the storage type).
//
// One CTA = one 128-row query tile of one (batch, head); two CTAs per SM.
//   warps 0-3  softmax: thread i owns query row i (= TMEM lane i), so row
//              max / row sum need no shuffles; the score row lives in 128 registers
//              (setmaxnreg moves registers from the data-movement warpgroup to this one)
//   warp  4    TMA producer: Q once, then a ring of K / V tiles
//   warp  5    MMA issuer (one lane): S = Q K^T, O += P V; owns the TMEM allocation
//   warps 6-7  idle (they complete the second warpgroup for setmaxnreg)
// TMEM columns (fp32): S [0,128)  P [128,192) (bf16 pairs)  O [192,256).
// Q, K, V are read straight from the projection output [B, N, H*64] through
// 4-D tensor maps (128-byte swizzle), so no head transpose is ever materialised.
#include <cuda.h>
#include <type_traits>
#include "common.cuh"
#include "ptx.cuh"

namespace mvoc {
namespace attn {

constexpr int BM = 128;  // query rows per CTA
constexpr int HD = 64;   // head dim
constexpr int Q_BYTES = BM * HD * 2;  // 16 KB: 128 rows x 128 B
constexpr int THREADS = 256;  // warps 0-3 softmax (warpgroup 0); 4 TMA, 5 MMA, 6-7 idle (warpgroup 1)
constexpr uint32_t TMEM_COLS = 256;
constexpr float RESCALE_LOG2_THRESHOLD = 8.0f;

// kBN keys per iteration, kNV value tensors sharing one softmax.  TMEM columns (fp32): S [0, kBN), P [kBN, 1.5 kBN)
// (16-bit pairs), O_v [1.5 kBN + 64 v, +64).
template <int kBN, int kNV, int kStages>
struct Smem {
    static constexpr int KV_BYTES = kBN * HD * 2;
    static constexpr int q_off = 0;
    static constexpr int k_off = Q_BYTES;
    static constexpr int v_off = k_off + kStages * KV_BYTES;
    static constexpr int bar_off = v_off + kStages * kNV * KV_BYTES;
    // barriers: q_full, s_full, s_free, p_full, pv_done, k_full[], k_empty[], v_full[], v_empty[]
    static constexpr int n_bars = 5 + 4 * kStages;
    static constexpr int tmem_ptr_off = bar_off + n_bars * 8;
    static constexpr int total = tmem_ptr_off + 16;
    // No alignment slack: the dynamic window is declared __align__(1024) and checked at run time.  Two CTAs
    // must fit one SM: 2 * (alloc + 1 KB reserved) <= 228 KB — with the 3-stage ring that leaves < 2 KB.
    static constexpr int alloc = total;
    static constexpr uint32_t COL_S = 0, COL_P = kBN, COL_O = kBN + kBN / 2;
    static_assert(2 * (alloc + 1024) <= 233472, "two CTAs per SM no longer fit in shared memory");
    static_assert(COL_O + 64 * kNV <= TMEM_COLS, "S + P + O accumulators exceed the CTA's TMEM columns");
    static_assert(kBN == 64 || kBN == 128, "key block of 64 or 128");
};

struct Params {
    void* o;
    int64_t o_sb, o_sn, o_sh;
    int Nq, Nk;
    int pair_batches;   // kNV == 2: the second value / output tensor is this many batches after the first
    float scale_log2;
    long long* trace;   // diagnostics (mvoc_attn_fwd_trace): clock64() of CTA (0,0,0) at 8 points per key block, or null
};

// trace slot layout: [block j][event]; events 0-5 by softmax thread 0, 6-7 by the MMA lane
__device__ __forceinline__ void trace_at(const Params& prm, int j, int ev) {
    if (prm.trace != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0) prm.trace[j * 8 + ev] = clock64();
}

// kEmuMask: bit (k % 8) set => the k-th pair of a score row takes the FMA-pipe exp2 instead of the MUFU.
template <typename T, int kBN, int kNV, int kStages, uint32_t kEmuMask, bool kCausal>
__global__ void __launch_bounds__(THREADS, 2)
attn_fwd_kernel(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_k,
                const __grid_constant__ CUtensorMap tm_v, const Params prm) {
    using L = Smem<kBN, kNV, kStages>;
    constexpr int BN = kBN;
    constexpr int KV_BYTES = L::KV_BYTES;
    constexpr uint32_t COL_S = L::COL_S, COL_P = L::COL_P, COL_O = L::COL_O;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const uint32_t sbase = smem_u32(smem_raw);
    uint8_t* sgen = smem_raw;
    MVOC_REQUIRE_SMEM_1024(sbase, "attn_fwd_kernel");

    const uint32_t sQ = sbase + L::q_off;
    const uint32_t sK = sbase + L::k_off;
    const uint32_t sV = sbase + L::v_off;
    const uint32_t bars = sbase + L::bar_off;
    const uint32_t b_q_full = bars, b_s_full = bars + 8, b_s_free = bars + 16, b_p_full = bars + 24,
                   b_pv_done = bars + 32;
    const uint32_t b_k_full = bars + 40, b_k_empty = b_k_full + 8 * kStages,
                   b_v_full = b_k_empty + 8 * kStages, b_v_empty = b_v_full + 8 * kStages;
    const uint32_t s_tmem_ptr = sbase + L::tmem_ptr_off;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m_blk = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
    static_assert(!kCausal || (kBN == BM && kNV == 1), "causal mode: plain attention on 128-key blocks");
    // causal: query tile m_blk needs key blocks 0..m_blk only (the host checks Nq == Nk)
    const int n_blocks = kCausal ? min((prm.Nk + BN - 1) / BN, m_blk + 1) : (prm.Nk + BN - 1) / BN;

    if (warp == 4 && lane == 0) {
        ptx::prefetch_tensormap(&tm_q);
        ptx::prefetch_tensormap(&tm_k);
        ptx::prefetch_tensormap(&tm_v);
        ptx::mbar_init(b_q_full, 1);
        ptx::mbar_init(b_s_full, 1);
        ptx::mbar_init(b_s_free, 4);     // one arrival per softmax warp (an elected lane after __syncwarp): 128
        ptx::mbar_init(b_p_full, 4);     // per-thread arrivals serialise on the barrier word in front of the MMA warp
        ptx::mbar_init(b_pv_done, 1);
        for (int s = 0; s < kStages; ++s) {
            ptx::mbar_init(b_k_full + 8 * s, 1);
            ptx::mbar_init(b_k_empty + 8 * s, 1);
            ptx::mbar_init(b_v_full + 8 * s, 1);
            ptx::mbar_init(b_v_empty + 8 * s, 1);
        }
        ptx::fence_mbar_init();
    }
    if (warp == 5) {
        ptx::tmem_alloc(s_tmem_ptr, TMEM_COLS);
        ptx::tmem_relinquish();
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem = *reinterpret_cast<volatile uint32_t*>(sgen + L::tmem_ptr_off);

    // Register re-allocation between the warpgroups: 2 CTAs/SM leave 128 registers per thread at launch;
    // the data-movement warpgroup keeps 48 and hands the rest to the softmax warpgroup, which needs the
    // whole 128-column score row in registers (208 each: 128*208 + 128*48 = 256*128).
    if (warp >= 4) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 48;" ::: "memory");
    if (warp == 4) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            ptx::mbar_expect_tx(b_q_full, Q_BYTES);
            ptx::tma_load_4d(sQ, &tm_q, b_q_full, 0, h, m_blk * BM, b);
        }
        for (int j = 0; j < n_blocks; ++j) {
            const int s = j % kStages;
            const uint32_t ph = (uint32_t)(j / kStages) & 1u;
            ptx::mbar_wait(b_k_empty + 8 * s, ph ^ 1u, 1);
            if (lane == 0) {
                ptx::mbar_expect_tx(b_k_full + 8 * s, KV_BYTES);
                ptx::tma_load_4d(sK + s * KV_BYTES, &tm_k, b_k_full + 8 * s, 0, h, j * BN, b);
            }
            ptx::mbar_wait(b_v_empty + 8 * s, ph ^ 1u, 2);
            if (lane == 0) {
                ptx::mbar_expect_tx(b_v_full + 8 * s, kNV * KV_BYTES);
#pragma unroll
                for (int v = 0; v < kNV; ++v)
                    ptx::tma_load_4d(sV + (s * kNV + v) * KV_BYTES, &tm_v, b_v_full + 8 * s, 0, h, j * BN,
                                     b + v * prm.pair_batches);
            }
            __syncwarp();
        }
    } else if (warp == 5) {
        // ===================== MMA issuer =====================
        constexpr bool kF16 = std::is_same<T, __half>::value;
        constexpr uint32_t IDESC_QK = ptx::idesc_f16(kF16, BM, BN, false);  // A,B K-major
        constexpr uint32_t IDESC_PV = ptx::idesc_f16(kF16, BM, HD, true);   // B (=V) MN-major
        const uint32_t tS = tmem + COL_S, tP = tmem + COL_P, tO = tmem + COL_O;
        auto issue_qk = [&](int j) {
            const int s = j % kStages;
            const uint64_t a0 = ptx::smem_desc_sw128(sQ, 16, 1024);
            const uint64_t b0 = ptx::smem_desc_sw128(sK + s * KV_BYTES, 16, 1024);
#pragma unroll
            for (int ks = 0; ks < HD / 16; ++ks)  // +32 B per 16-element K step (encoded >>4)
                ptx::mma_ss(tS, a0 + (uint64_t)(ks * 2), b0 + (uint64_t)(ks * 2), IDESC_QK, ks > 0);
            ptx::tc_commit(b_k_empty + 8 * s);
            ptx::tc_commit(b_s_full);
        };
        ptx::mbar_wait(b_q_full, 0, 3);
        ptx::mbar_wait(b_k_full, 0, 4);
        ptx::tc_fence_after();
        if (lane == 0) issue_qk(0);
        __syncwarp();
        for (int j = 0; j < n_blocks; ++j) {
            const int s = j % kStages;
            const uint32_t ph = (uint32_t)(j / kStages) & 1u;
            if (j + 1 < n_blocks) {
                const int s1 = (j + 1) % kStages;
                ptx::mbar_wait(b_k_full + 8 * s1, (uint32_t)((j + 1) / kStages) & 1u, 5);
                ptx::mbar_wait(b_s_free, (uint32_t)j & 1u, 6);
                ptx::tc_fence_after();
                if (lane == 0) {
                    issue_qk(j + 1);
                    trace_at(prm, j + 1, 6);   // Q K^T of block j+1 issued
                }
                __syncwarp();
            }
            ptx::mbar_wait(b_v_full + 8 * s, ph, 7);
            ptx::mbar_wait(b_p_full, (uint32_t)j & 1u, 8);
            ptx::tc_fence_after();
            if (lane == 0) {
                // V tile: rows = keys (K of this GEMM), 128 B per row = 64 d (N) contiguous
#pragma unroll
                for (int v = 0; v < kNV; ++v) {
                    const uint64_t bv = ptx::smem_desc_sw128(sV + (s * kNV + v) * KV_BYTES, 16384, 1024);
#pragma unroll
                    for (int ks = 0; ks < BN / 16; ++ks)
                        ptx::mma_ts(tO + v * HD, tP + ks * 8, bv + (uint64_t)((ks * 2048) >> 4), IDESC_PV,
                                    (j > 0 || ks > 0) ? 1u : 0u);
                }
                ptx::tc_commit(b_v_empty + 8 * s);
                ptx::tc_commit(b_pv_done);
                trace_at(prm, j, 7);           // P V of block j issued
            }
            __syncwarp();
        }
    }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 208;" ::: "memory");
        // ===================== softmax + epilogue (warps 0-3) =====================
        const int row = threadIdx.x;  // query row inside the tile == TMEM lane
        const uint32_t lane_base = tmem + ((uint32_t)(warp * 32) << 16);
        const uint32_t tS = lane_base + COL_S, tP = lane_base + COL_P, tO = lane_base + COL_O;
        const float sl2 = prm.scale_log2;
        float m_used = -INFINITY, l_sum = 0.0f;
        bool s_ready = false;   // S of the next block already seen complete by a non-blocking poll
        for (int j = 0; j < n_blocks; ++j) {
            // causal: in the diagonal block, column i is key m_blk*BM + i and must not exceed query row m_blk*BM + row
            const int valid = kCausal && j == m_blk ? min(min(BN, prm.Nk - j * BN), row + 1) : min(BN, prm.Nk - j * BN);
            const bool tail = valid < BN;
            if (threadIdx.x == 0) trace_at(prm, j, 0);   // softmax of block j starts waiting for S
            if (!s_ready) ptx::mbar_wait(b_s_full, (uint32_t)j & 1u, 9);
            ptx::tc_fence_after();
            if (threadIdx.x == 0) trace_at(prm, j, 1);   // S ready
            // One TMEM read of the whole score row (BN fp32 columns -> BN registers); S is free for the next
            // Q K^T as soon as it sits in registers, long before the exponentials are done.  (Measured on B200:
            // reading and reducing the row in 32-column pieces, with or without exponentiating each piece at once,
            // is slower — 2.27 / 2.31 ms against 2.04 ms at the l0 shape: the waits between the pieces serialise what
            // the scheduler otherwise overlaps across the 64 independent pairs of the row.)
            uint32_t r[BN];
#pragma unroll
            for (int c = 0; c < BN / 32; ++c)
                ptx::tmem_ld32(tS + c * 32, *reinterpret_cast<uint32_t(*)[32]>(&r[c * 32]));
            ptx::tmem_wait_ld();
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(b_s_free);
            if (tail) {  // keys past Nk (zero-filled by TMA) or, causal, past the row must not take part: exp2(-inf) = 0
#pragma unroll
                for (int i = 0; i < BN; ++i)
                    if (i >= valid) r[i] = 0xff800000u;
            }
            // row max: eight independent chains of 3-input max (FMNMX3), 8 deep for a 128-column row
            float mxc[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) mxc[e] = -INFINITY;
#pragma unroll
            for (int i = 0; i < BN; i += 16) {
#pragma unroll
                for (int e = 0; e < 8; ++e)
                    mxc[e] = ptx::max3(mxc[e], __uint_as_float(r[i + 2 * e]), __uint_as_float(r[i + 2 * e + 1]));
            }
            const float mx = fmaxf(ptx::max3(mxc[0], mxc[1], mxc[2]), fmaxf(ptx::max3(mxc[3], mxc[4], mxc[5]), fmaxf(mxc[6], mxc[7])));
            bool pv_waited = false;            // the previous P V is known complete (blocking wait done)
            bool pv_ready = (j == 0);          // ... or seen complete by the non-blocking poll
            if (j == 0) {
                m_used = mx;
            } else {
                const float m_new = fmaxf(m_used, mx);
                const bool need = (m_new - m_used) * sl2 > RESCALE_LOG2_THRESHOLD;
                if (__any_sync(0xffffffffu, need)) {
                    // rescale the running O and l (rare after the first blocks)
                    ptx::mbar_wait(b_pv_done, (uint32_t)(j - 1) & 1u, 10);
                    ptx::tc_fence_after();
                    pv_waited = true;
                    const float f = need ? ptx::ex2_approx((m_used - m_new) * sl2) : 1.0f;
                    if (need) m_used = m_new;
                    l_sum *= f;
#pragma unroll
                    for (int c = 0; c < kNV * HD / 32; ++c) {
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
            if (threadIdx.x == 0) trace_at(prm, j, 2);   // row in registers, maximum known, rescale decided
            // p = exp2(s * scale*log2e - m * scale*log2e) on pairs (FFMA2); the exponential goes to the MUFU or,
            // for the pairs selected by kEmuMask, to the FMA-pipe polynomial; packed row sums (FADD2).
            const uint64_t sl2_2 = ptx::pack2(sl2, sl2);
            const uint64_t negm_2 = ptx::pack2(-m_used * sl2, -m_used * sl2);
            uint32_t pk[BN / 2];
            uint64_t la = ptx::pack2(0.0f, 0.0f), lb = la, lc = la, ld = la;
#pragma unroll
            for (int k = 0; k < BN / 2; ++k) {
                const uint64_t x2 = ptx::fma2(ptx::pack2(__uint_as_float(r[2 * k]), __uint_as_float(r[2 * k + 1])),
                                              sl2_2, negm_2);
                float p0, p1;
                if ((kEmuMask >> (k & 7)) & 1u) {
                    ptx::ex2_poly2(x2, p0, p1);
                } else {
                    float x0, x1;
                    ptx::unpack2(x2, x0, x1);
                    p0 = ptx::ex2_approx(x0);
                    p1 = ptx::ex2_approx(x1);
                }
                const uint64_t p2 = ptx::pack2(p0, p1);
                if ((k & 3) == 0) la = ptx::add2(la, p2);
                else if ((k & 3) == 1) lb = ptx::add2(lb, p2);
                else if ((k & 3) == 2) lc = ptx::add2(lc, p2);
                else ld = ptx::add2(ld, p2);
                pk[k] = pack2_rn<T>(p0, p1);
                // two thirds through: poll (without blocking) whether the previous P V has completed, so that the wait
                // in front of the P store costs nothing when it has (an mbarrier wait costs ~130 clocks even then)
                if (k == (BN / 2) * 2 / 3 && !pv_waited && !pv_ready)
                    pv_ready = ptx::mbar_test(b_pv_done, (uint32_t)(j - 1) & 1u);
            }
            {
                float s0, s1;
                ptx::unpack2(ptx::add2(ptx::add2(la, lb), ptx::add2(lc, ld)), s0, s1);
                l_sum += s0 + s1;
            }
            if (threadIdx.x == 0) trace_at(prm, j, 3);   // exponentials done
            // P buffer is free once the previous P V has completed
            if (!pv_waited) {
                if (!pv_ready) ptx::mbar_wait(b_pv_done, (uint32_t)(j - 1) & 1u, 11);
                ptx::tc_fence_after();
            }
            if (threadIdx.x == 0) trace_at(prm, j, 4);   // previous P V complete (P buffer free)
#pragma unroll
            for (int c = 0; c < BN / 64; ++c)
                ptx::tmem_st32(tP + c * 32, *reinterpret_cast<uint32_t(*)[32]>(&pk[c * 32]));
            // while the P store drains: has the next Q K^T already landed?
            s_ready = (j + 1 < n_blocks) && ptx::mbar_test(b_s_full, (uint32_t)(j + 1) & 1u);
            ptx::tmem_wait_st();
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(b_p_full);
            if (threadIdx.x == 0) trace_at(prm, j, 5);   // P published
        }
        // ---- epilogue: O / l -> 16-bit -> global --------------------------------
        ptx::mbar_wait(b_pv_done, (uint32_t)(n_blocks - 1) & 1u, 12);
        ptx::tc_fence_after();
        const float inv_l = 1.0f / l_sum;
        const int q_row = m_blk * BM + row;
#pragma unroll
        for (int v = 0; v < kNV; ++v) {
            T* orow = reinterpret_cast<T*>(prm.o) + (int64_t)(b + v * prm.pair_batches) * prm.o_sb +
                      (int64_t)q_row * prm.o_sn + (int64_t)h * prm.o_sh;
#pragma unroll
            for (int c = 0; c < HD / 32; ++c) {
                uint32_t r[32];
                ptx::tmem_ld32(tO + v * HD + c * 32, r);
                ptx::tmem_wait_ld();
                if (q_row < prm.Nq) {
#pragma unroll
                    for (int i = 0; i < 32; i += 8) {
                        float f[8];
#pragma unroll
                        for (int e = 0; e < 8; ++e) f[e] = __uint_as_float(r[i + e]) * inv_l;
                        *reinterpret_cast<Vec16*>(orow + c * 32 + i) = pack8<T>(f);
                    }
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
template <typename T, int kBN, int kNV, int kStages, uint32_t kEmuMask, bool kCausal = false>
static int launch(const CUtensorMap (&m)[3], const Params& prm, int B, int H, cudaStream_t s, const char* what) {
    using L = Smem<kBN, kNV, kStages>;
    static bool smem_set[64] = {false};
    const int rc = set_max_dynamic_smem((const void*)attn_fwd_kernel<T, kBN, kNV, kStages, kEmuMask, kCausal>, L::alloc,
                                        smem_set, what);
    if (rc != MVOC_OK) return rc;
    dim3 grid((prm.Nq + BM - 1) / BM, H, B);
    attn_fwd_kernel<T, kBN, kNV, kStages, kEmuMask, kCausal><<<grid, THREADS, L::alloc, s>>>(m[0], m[1], m[2], prm);
    return check_launch(what);
}

// Common entry: kNV value tensors per softmax (1 = plain attention, 2 = the uncond/cond pair).
// causal: plain attention only (pair_batches == 0, variant 0), Nq == Nk.
static int run(const void* q, const void* k, const void* v, void* o, int B, int H, int Nq, int Nk, int D,
               const int64_t (&st)[12], int pair_batches, float scale, int dtype, int variant, void* stream,
               const char* what, long long* trace = nullptr, bool causal = false) {
    int rc = check_attn_operands(q, k, v, o, dtype, D, HD, st, 12, what);
    if (rc != MVOC_OK) return rc;
    MVOC_REQUIRE(B > 0 && H > 0 && Nq > 0 && Nk > 0, MVOC_ERR_INVALID_ARG, "%s: empty problem B=%d H=%d Nq=%d Nk=%d", what,
                 B, H, Nq, Nk);
    MVOC_REQUIRE(B <= 65535 && H <= 65535, MVOC_ERR_UNSUPPORTED, "%s: B=%d / H=%d exceed the grid limits", what, B, H);
    MVOC_REQUIRE(variant >= 0 && variant <= 5, MVOC_ERR_INVALID_ARG, "%s: unknown variant %d", what, variant);
    MVOC_REQUIRE(pair_batches >= 0, MVOC_ERR_INVALID_ARG, "%s: pair_batches=%d", what, pair_batches);
    MVOC_REQUIRE(!causal || Nq == Nk, MVOC_ERR_UNSUPPORTED, "%s: causal attention needs Nq == Nk, got Nq=%d Nk=%d",
                 what, Nq, Nk);
    const bool pair = pair_batches > 0;
    const int kv_rows = pair ? 64 : 128;
    // q, k, v: [B, N, H, 64] viewed innermost first with element strides (sh, sn, sb); box = one head's 64 columns of
    // `rows` tokens
    const void* ptr[3] = {q, k, v};
    const char* name[3] = {"q", "k", "v"};
    const int64_t dims[3][4] = {{HD, H, Nq, B}, {HD, H, Nk, B}, {HD, H, Nk, B + pair_batches}};
    const int64_t str[3][3] = {{st[2], st[1], st[0]}, {st[5], st[4], st[3]}, {st[8], st[7], st[6]}};
    const int rows[3] = {BM, kv_rows, kv_rows};
    for (int i = 0; i < 3; ++i)   // all three before the first driver call
        if ((rc = check_map4(dims[i], str[i], what, name[i])) != MVOC_OK) return rc;
    // CTA b writes O[b] and O[b + pair_batches]: below B, a second output batch is also written by another CTA
    MVOC_REQUIRE(!pair || pair_batches >= B, MVOC_ERR_INVALID_ARG, "%s: pair_batches=%d < B=%d", what, pair_batches, B);
    CUtensorMap m[3];
    for (int i = 0; i < 3; ++i) {
        const int box[4] = {HD, 1, rows[i], 1};
        if ((rc = make_map4(&m[i], ptr[i], dtype, dims[i], str[i], box, 1, CU_TENSOR_MAP_SWIZZLE_128B, what, name[i])) !=
            MVOC_OK)
            return rc;
    }
    Params prm;
    prm.o = o;
    prm.o_sb = st[9];
    prm.o_sn = st[10];
    prm.o_sh = st[11];
    prm.Nq = Nq;
    prm.Nk = Nk;
    prm.pair_batches = pair_batches;
    prm.scale_log2 = scale * 1.4426950408889634f;
    prm.trace = trace;
    cudaStream_t s = (cudaStream_t)stream;
    if (causal) {
        if (dtype == MVOC_F16) return launch<__half, 128, 1, 3, 0xA8u, true>(m, prm, B, H, s, what);
        return launch<__nv_bfloat16, 128, 1, 3, 0xA8u, true>(m, prm, B, H, s, what);
    }
    // variants (same results up to the exp2 approximation; the tests run all of them):
    //   1, 2: all exponentials on the MUFU;  3 / 4 / 5: 2 / 3 / 4 of every 8 pairs on the FMA-pipe polynomial;  0: default
    const uint32_t emu = variant == 1 || variant == 2 ? 0x00u : variant == 3 ? 0x88u : variant == 5 ? 0xAAu : 0xA8u;
#define MVOC_ATTN_LAUNCH(T, BN, NV, EMU) launch<T, BN, NV, 3, EMU>(m, prm, B, H, s, what)
#define MVOC_ATTN_EMU(T, BN, NV)                                           \
    switch (emu) {                                                         \
        case 0x00u: return MVOC_ATTN_LAUNCH(T, BN, NV, 0x00u);             \
        case 0x88u: return MVOC_ATTN_LAUNCH(T, BN, NV, 0x88u);             \
        case 0xAAu: return MVOC_ATTN_LAUNCH(T, BN, NV, 0xAAu);             \
        default: return MVOC_ATTN_LAUNCH(T, BN, NV, 0xA8u); /* fastest measured on B200 */ \
    }
    if (dtype == MVOC_F16) {
        if (pair) { MVOC_ATTN_EMU(__half, 64, 2) }
        MVOC_ATTN_EMU(__half, 128, 1)
    }
    if (pair) { MVOC_ATTN_EMU(__nv_bfloat16, 64, 2) }
    MVOC_ATTN_EMU(__nv_bfloat16, 128, 1)
#undef MVOC_ATTN_EMU
#undef MVOC_ATTN_LAUNCH
}

}  // namespace attn

int check_attn_operands(const void* q, const void* k, const void* v, const void* o, int dtype, int D, int head_dim,
                        const int64_t* st, int n_st, const char* what) {
    MVOC_REQUIRE(q && k && v && o, MVOC_ERR_INVALID_ARG, "%s: null pointer", what);
    MVOC_REQUIRE(dtype == MVOC_BF16 || dtype == MVOC_F16, MVOC_ERR_UNSUPPORTED, "%s: dtype %d unsupported (bf16 / fp16)",
                 what, dtype);
    MVOC_REQUIRE(D == head_dim, MVOC_ERR_UNSUPPORTED, "%s: head_dim %d unsupported (%d only)", what, D, head_dim);
    for (int i = 0; i < n_st; ++i)
        MVOC_REQUIRE(st[i] % 8 == 0 && st[i] >= 0, MVOC_ERR_UNSUPPORTED,
                     "%s: stride #%d = %lld is not a non-negative multiple of 8 elements", what, i, (long long)st[i]);
    MVOC_REQUIRE(((uintptr_t)q % 16 == 0) && ((uintptr_t)k % 16 == 0) && ((uintptr_t)v % 16 == 0) &&
                     ((uintptr_t)o % 16 == 0),
                 MVOC_ERR_INVALID_ARG, "%s: pointers must be 16-byte aligned", what);
    return MVOC_OK;
}

}  // namespace mvoc

using namespace mvoc;

extern "C" int mvoc_attn_fwd(const void* q, const void* k, const void* v, void* o, int B, int H,
                             int Nq, int Nk, int D, int64_t q_sb, int64_t q_sn, int64_t q_sh,
                             int64_t k_sb, int64_t k_sn, int64_t k_sh, int64_t v_sb, int64_t v_sn,
                             int64_t v_sh, int64_t o_sb, int64_t o_sn, int64_t o_sh, float scale,
                             int dtype, int variant, void* stream) {
    const int64_t st[12] = {q_sb, q_sn, q_sh, k_sb, k_sn, k_sh, v_sb, v_sn, v_sh, o_sb, o_sn, o_sh};
    return attn::run(q, k, v, o, B, H, Nq, Nk, D, st, 0, scale, dtype, variant, stream, "mvoc_attn_fwd");
}

extern "C" int mvoc_attn_causal_fwd(const void* q, const void* k, const void* v, void* o, int B, int H, int Nq,
                                    int Nk, int D, int64_t q_sb, int64_t q_sn, int64_t q_sh, int64_t k_sb, int64_t k_sn,
                                    int64_t k_sh, int64_t v_sb, int64_t v_sn, int64_t v_sh, int64_t o_sb, int64_t o_sn,
                                    int64_t o_sh, float scale, int dtype, void* stream) {
    const int64_t st[12] = {q_sb, q_sn, q_sh, k_sb, k_sn, k_sh, v_sb, v_sn, v_sh, o_sb, o_sn, o_sh};
    return attn::run(q, k, v, o, B, H, Nq, Nk, D, st, 0, scale, dtype, 0, stream, "mvoc_attn_causal_fwd", nullptr,
                     true);
}

extern "C" int mvoc_attn_pair_fwd(const void* q, const void* k, const void* v, void* o, int B, int H,
                                  int Nq, int Nk, int D, int64_t q_sb, int64_t q_sn, int64_t q_sh,
                                  int64_t k_sb, int64_t k_sn, int64_t k_sh, int64_t v_sb, int64_t v_sn,
                                  int64_t v_sh, int64_t o_sb, int64_t o_sn, int64_t o_sh, int pair_batches,
                                  float scale, int dtype, int variant, void* stream) {
    const int64_t st[12] = {q_sb, q_sn, q_sh, k_sb, k_sn, k_sh, v_sb, v_sn, v_sh, o_sb, o_sn, o_sh};
    MVOC_REQUIRE(pair_batches > 0, MVOC_ERR_INVALID_ARG, "mvoc_attn_pair_fwd: pair_batches=%d must be positive",
                 pair_batches);
    return attn::run(q, k, v, o, B, H, Nq, Nk, D, st, pair_batches, scale, dtype, variant, stream, "mvoc_attn_pair_fwd");
}

// Diagnostics: mvoc_attn_fwd (or the pair kernel when pair_batches > 0) with clock64() time stamps of CTA (0,0,0):
// trace[j*8 + e] for key block j and event e — 0 softmax waits for S, 1 S ready, 2 maximum known, 3 exponentials
// done, 4 P buffer free, 5 P published (softmax thread 0); 6 Q K^T issued, 7 P V issued (MMA lane).
extern "C" int mvoc_attn_fwd_trace(const void* q, const void* k, const void* v, void* o, int B, int H, int Nq, int Nk,
                                   int D, const int64_t* strides12, int pair_batches, float scale, int dtype, int variant,
                                   long long* trace, void* stream) {
    MVOC_REQUIRE(strides12 && trace, MVOC_ERR_INVALID_ARG, "mvoc_attn_fwd_trace: null pointer");
    int64_t st[12];
    for (int i = 0; i < 12; ++i) st[i] = strides12[i];
    return attn::run(q, k, v, o, B, H, Nq, Nk, D, st, pair_batches, scale, dtype, variant, stream, "mvoc_attn_fwd_trace",
                     trace);
}
