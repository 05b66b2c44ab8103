// Short-sequence ("temporal") attention: tokens = frames (T <= 32), D = 64.
// Reference: F.scaled_dot_product_attention at i2vgen-xl/pnp_utils.py:862-864
// and the stock processor behind attention_forward (:348-385) for the
// temporal attn2 / transformer_in, all driven by
// transformer_temporal_model_forward (:170-220) on [(b h w), T, C] tensors.
//
// Arithmetic intensity is ~8 FLOP/B (read Q,K,V + write O once), so this is an
// HBM-bound kernel: one warp owns one (pixel, head) problem, pulls the three
// T x 64 bf16 tiles with 16-byte cp.async (full 128-byte lines), runs the two
// tiny GEMMs on mma.sync fragments (enough to stay under the memory time; a
// tcgen05 tile would be 87 % padding at T = 16), and writes O back through
// shared memory as full 128-byte rows.
#include "common.cuh"

namespace mvoc {

constexpr int TA_WARPS = 4;

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2,
                                        uint32_t& r3) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
                 : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2,
                                          uint32_t& r3) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
                 : "r"(addr));
}
__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2,
                                               uint32_t a3, uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, "
        "{%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
// byte offset of 16-byte chunk `c` of row `r` in a 128-byte-row, XOR-swizzled tile
__device__ __forceinline__ uint32_t swz(int r, int c) { return (uint32_t)(r * 128 + ((c ^ (r & 7)) << 4)); }

struct TAParams {
    const __nv_bfloat16 *q, *k, *v;
    __nv_bfloat16* o;
    int64_t P;        // problems = P_outer * P_inner
    int64_t P_inner;  // problem index = outer * P_inner + inner
    int H;
    int T;
    // element strides: (outer problem, inner problem, token, head) per tensor
    int64_t q_so, q_sp, q_st, q_sh, k_so, k_sp, k_st, k_sh, v_so, v_sp, v_st, v_sh, o_so, o_sp, o_st, o_sh;
    float scale_log2;
};

// TP = rows held in smem (16 or 32); kExact: T == TP (no masking, fully unrolled loads).
template <int TP, bool kExact>
__global__ void __launch_bounds__(TA_WARPS * 32) attn_temporal_kernel(TAParams p) {
    constexpr int MT = TP / 16;         // query m-tiles
    constexpr int NT = TP / 8;          // key n-tiles
    constexpr int KT = MT;              // PV k-steps of 16 keys
    constexpr int TILE = TP * 128;      // bytes per matrix
    const int T = kExact ? TP : p.T;    // frames actually present
    extern __shared__ __align__(128) uint8_t ta_smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t item = (int64_t)blockIdx.x * TA_WARPS + warp;
    if (item >= p.P * p.H) return;
    const int64_t prob = item / p.H;
    const int h = (int)(item % p.H);
    const uint32_t sQ = smem_u32(ta_smem) + warp * 3 * TILE, sK = sQ + TILE, sV = sK + TILE;

    const int64_t po = prob / p.P_inner, pi = prob - po * p.P_inner;
    const __nv_bfloat16* gq = p.q + po * p.q_so + pi * p.q_sp + (int64_t)h * p.q_sh;
    const __nv_bfloat16* gk = p.k + po * p.k_so + pi * p.k_sp + (int64_t)h * p.k_sh;
    const __nv_bfloat16* gv = p.v + po * p.v_so + pi * p.v_sp + (int64_t)h * p.v_sh;
    if (kExact) {
#pragma unroll
        for (int i = 0; i < (TP * 8) / 32; ++i) {
            const int idx = lane + 32 * i, r = idx >> 3, c = idx & 7;
            cp_async16(sQ + swz(r, c), gq + (int64_t)r * p.q_st + c * 8);
            cp_async16(sK + swz(r, c), gk + (int64_t)r * p.k_st + c * 8);
            cp_async16(sV + swz(r, c), gv + (int64_t)r * p.v_st + c * 8);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    } else {
        for (int idx = lane; idx < T * 8; idx += 32) {
            const int r = idx >> 3, c = idx & 7;
            cp_async16(sQ + swz(r, c), gq + (int64_t)r * p.q_st + c * 8);
            cp_async16(sK + swz(r, c), gk + (int64_t)r * p.k_st + c * 8);
            cp_async16(sV + swz(r, c), gv + (int64_t)r * p.v_st + c * 8);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        // zero the padding rows: Q rows give harmless uniform rows that are never stored, K rows are masked
        // below, V rows must be finite because they meet P = 0
        const Vec16 z = {{0u, 0u, 0u, 0u}};
        for (int idx = lane; idx < (TP - T) * 8; idx += 32) {
            const int r = T + (idx >> 3), c = idx & 7;
            uint8_t* base = ta_smem + warp * 3 * TILE;
            *reinterpret_cast<Vec16*>(base + swz(r, c)) = z;
            *reinterpret_cast<Vec16*>(base + TILE + swz(r, c)) = z;
            *reinterpret_cast<Vec16*>(base + 2 * TILE + swz(r, c)) = z;
        }
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncwarp();

    const int g = lane >> 2, t = lane & 3;
    const int mat = lane >> 3, mr = lane & 7;
    __nv_bfloat16* go = p.o + po * p.o_so + pi * p.o_sp + (int64_t)h * p.o_sh;

#pragma unroll
    for (int mt = 0; mt < MT; ++mt) {
        // ---- S = Q K^T for this m-tile -----------------------------------
        float s[NT][4];
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.0f;
#pragma unroll
        for (int ks = 0; ks < 4; ks += 2) {
            uint32_t a[2][4];
#pragma unroll
            for (int kk = 0; kk < 2; ++kk) {
                const int row = mt * 16 + (mat & 1) * 8 + mr;
                const int chunk = 2 * (ks + kk) + (mat >> 1);
                ldsm_x4(sQ + swz(row, chunk), a[kk][0], a[kk][1], a[kk][2], a[kk][3]);
            }
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                uint32_t b0, b1, b2, b3;
                ldsm_x4(sK + swz(nt * 8 + mr, 2 * ks + mat), b0, b1, b2, b3);
                mma_bf16_16816(s[nt], a[0][0], a[0][1], a[0][2], a[0][3], b0, b1);
                mma_bf16_16816(s[nt], a[1][0], a[1][1], a[1][2], a[1][3], b2, b3);
            }
        }
        if (!kExact) {  // keys >= T do not exist
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                const int key = nt * 8 + 2 * t;
                if (key >= T) s[nt][0] = s[nt][2] = -INFINITY;
                if (key + 1 >= T) s[nt][1] = s[nt][3] = -INFINITY;
            }
        }
        // ---- softmax over keys (rows g and g+8 of the tile) ---------------
        float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            m0 = fmaxf(m0, fmaxf(s[nt][0], s[nt][1]));
            m1 = fmaxf(m1, fmaxf(s[nt][2], s[nt][3]));
        }
        m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1));
        m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
        m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1));
        m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
        const float o0 = -m0 * p.scale_log2, o1 = -m1 * p.scale_log2;
        float l0 = 0.0f, l1 = 0.0f;
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            s[nt][0] = exp2f(fmaf(s[nt][0], p.scale_log2, o0));
            s[nt][1] = exp2f(fmaf(s[nt][1], p.scale_log2, o0));
            s[nt][2] = exp2f(fmaf(s[nt][2], p.scale_log2, o1));
            s[nt][3] = exp2f(fmaf(s[nt][3], p.scale_log2, o1));
            l0 += s[nt][0] + s[nt][1];
            l1 += s[nt][2] + s[nt][3];
        }
        l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
        l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
        l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
        l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
        // ---- O = P V ------------------------------------------------------
        float o[8][4];
#pragma unroll
        for (int dn = 0; dn < 8; ++dn) o[dn][0] = o[dn][1] = o[dn][2] = o[dn][3] = 0.0f;
#pragma unroll
        for (int kk = 0; kk < KT; ++kk) {
            const uint32_t a0 = pack2_rn<__nv_bfloat16>(s[2 * kk][0], s[2 * kk][1]);
            const uint32_t a1 = pack2_rn<__nv_bfloat16>(s[2 * kk][2], s[2 * kk][3]);
            const uint32_t a2 = pack2_rn<__nv_bfloat16>(s[2 * kk + 1][0], s[2 * kk + 1][1]);
            const uint32_t a3 = pack2_rn<__nv_bfloat16>(s[2 * kk + 1][2], s[2 * kk + 1][3]);
#pragma unroll
            for (int dn = 0; dn < 8; dn += 2) {
                uint32_t b0, b1, b2, b3;
                ldsm_x4_t(sV + swz(16 * kk + (mat & 1) * 8 + mr, dn + (mat >> 1)), b0, b1, b2, b3);
                mma_bf16_16816(o[dn], a0, a1, a2, a3, b0, b1);
                mma_bf16_16816(o[dn + 1], a0, a1, a2, a3, b2, b3);
            }
        }
        // ---- normalise, stage in the Q rows of this m-tile, write out ------
        const float i0 = 1.0f / l0, i1 = 1.0f / l1;
        uint8_t* stage = ta_smem + warp * 3 * TILE;
        __syncwarp();
#pragma unroll
        for (int dn = 0; dn < 8; ++dn) {
            *reinterpret_cast<uint32_t*>(stage + swz(mt * 16 + g, dn) + t * 4) =
                pack2_rn<__nv_bfloat16>(o[dn][0] * i0, o[dn][1] * i0);
            *reinterpret_cast<uint32_t*>(stage + swz(mt * 16 + g + 8, dn) + t * 4) =
                pack2_rn<__nv_bfloat16>(o[dn][2] * i1, o[dn][3] * i1);
        }
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int idx = lane + 32 * i, r = mt * 16 + (idx >> 3), c = idx & 7;
            if (r < T) {
                const Vec16 v = *reinterpret_cast<const Vec16*>(stage + swz(r, c));
                st_stream16(go + (int64_t)r * p.o_st + c * 8, v);
            }
        }
    }
}

template <int TP, bool kExact>
static int ta_launch(const TAParams& p, cudaStream_t s) {
    const size_t smem = (size_t)TA_WARPS * 3 * TP * 128;
    const int64_t items = p.P * p.H;
    const int64_t grid = (items + TA_WARPS - 1) / TA_WARPS;
    attn_temporal_kernel<TP, kExact><<<(unsigned)grid, TA_WARPS * 32, smem, s>>>(p);
    return check_launch("mvoc_attn_temporal_fwd");
}

}  // namespace mvoc

using namespace mvoc;

static int ta_dispatch(const char* name, const void* q, const void* k, const void* v, void* o,
                       int64_t P_outer, int64_t P_inner, int T, int H, int D, const int64_t* st /*[16]*/,
                       float scale, int dtype, void* stream) {
    MVOC_REQUIRE(q && k && v && o, MVOC_ERR_INVALID_ARG, "%s: null pointer", name);
    MVOC_REQUIRE(dtype == MVOC_BF16, MVOC_ERR_UNSUPPORTED, "%s: dtype %d unsupported (bf16 only)", name, dtype);
    MVOC_REQUIRE(D == 64, MVOC_ERR_UNSUPPORTED, "%s: head_dim %d unsupported (64 only)", name, D);
    MVOC_REQUIRE(P_outer >= 0 && P_inner > 0 && H > 0, MVOC_ERR_INVALID_ARG, "%s: bad P/H", name);
    const int64_t P = P_outer * P_inner;
    MVOC_REQUIRE(P * H < ((int64_t)1 << 31) * TA_WARPS, MVOC_ERR_UNSUPPORTED, "%s: too many problems", name);
    for (int i = 0; i < 16; ++i)
        MVOC_REQUIRE(st[i] % 8 == 0, MVOC_ERR_UNSUPPORTED,
                     "%s: stride #%d = %lld is not a multiple of 8 elements", name, i, (long long)st[i]);
    MVOC_REQUIRE(((uintptr_t)q % 16 == 0) && ((uintptr_t)k % 16 == 0) && ((uintptr_t)v % 16 == 0) &&
                     ((uintptr_t)o % 16 == 0),
                 MVOC_ERR_INVALID_ARG, "%s: pointers must be 16-byte aligned", name);
    if (P == 0) return MVOC_OK;
    TAParams p;
    p.q = (const __nv_bfloat16*)q;
    p.k = (const __nv_bfloat16*)k;
    p.v = (const __nv_bfloat16*)v;
    p.o = (__nv_bfloat16*)o;
    p.P = P;
    p.P_inner = P_inner;
    p.H = H;
    p.q_so = st[0]; p.q_sp = st[1]; p.q_st = st[2]; p.q_sh = st[3];
    p.k_so = st[4]; p.k_sp = st[5]; p.k_st = st[6]; p.k_sh = st[7];
    p.v_so = st[8]; p.v_sp = st[9]; p.v_st = st[10]; p.v_sh = st[11];
    p.o_so = st[12]; p.o_sp = st[13]; p.o_st = st[14]; p.o_sh = st[15];
    p.scale_log2 = scale * 1.4426950408889634f;
    cudaStream_t s = (cudaStream_t)stream;
    p.T = T;
    if (T == 16) return ta_launch<16, true>(p, s);
    if (T == 32) return ta_launch<32, true>(p, s);
    if (T >= 1 && T < 16) return ta_launch<16, false>(p, s);
    if (T > 16 && T < 32) return ta_launch<32, false>(p, s);
    set_error("%s: T=%d unsupported (1..32 frames)", name, T);
    return MVOC_ERR_UNSUPPORTED;
}

extern "C" int mvoc_attn_temporal_fwd(const void* q, const void* k, const void* v, void* o,
                                      int64_t P, int T, int H, int D, int64_t q_sp, int64_t q_st,
                                      int64_t q_sh, int64_t k_sp, int64_t k_st, int64_t k_sh,
                                      int64_t v_sp, int64_t v_st, int64_t v_sh, int64_t o_sp,
                                      int64_t o_st, int64_t o_sh, float scale, int dtype,
                                      void* stream) {
    const int64_t st[16] = {0, q_sp, q_st, q_sh, 0, k_sp, k_st, k_sh, 0, v_sp, v_st, v_sh, 0, o_sp, o_st, o_sh};
    return ta_dispatch("mvoc_attn_temporal_fwd", q, k, v, o, P > 0 ? 1 : 0, P > 0 ? P : 1, T, H, D, st,
                       scale, dtype, stream);
}

extern "C" int mvoc_attn_temporal_strided_fwd(const void* q, const void* k, const void* v, void* o,
                                              int64_t P_outer, int64_t P_inner, int T, int H, int D,
                                              const int64_t* strides16, float scale, int dtype,
                                              void* stream) {
    MVOC_REQUIRE(strides16 != nullptr, MVOC_ERR_INVALID_ARG, "mvoc_attn_temporal_strided_fwd: null strides");
    return ta_dispatch("mvoc_attn_temporal_strided_fwd", q, k, v, o, P_outer, P_inner, T, H, D, strides16,
                       scale, dtype, stream);
}
