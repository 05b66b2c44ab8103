// GroupNorm (+SiLU) for NCHW activations, HBM-bound.
// Reference call sites: i2vgen-xl/pnp_utils.py:909-910, :953-965 (resnet
// norm1/norm2 + SiLU), :1048-1051 (TemporalConvLayer GN->SiLU heads), :430
// (Transformer2DModel.norm), :185-188 (TransformerTemporalModel.norm on the
// 5-D view), pipelines/pipeline_i2vgen_xl.py:351-352 (conv_norm_out + SiLU).
//
// Two paths:
//  A. smem-resident single pass (frames_per_stat == 1 and one (n, group) slab
//     fits in shared memory): the slab is pulled in with cp.async.bulk, mean
//     and centred variance are reduced from shared memory, the normalised
//     (+SiLU) values overwrite the slab and leave with one bulk store.
//     HBM traffic = 1 read + 1 write = the algorithmic 2*|X| bytes.
//  B. split statistics + apply (slabs too large for smem, or statistics that
//     span T frames of the [B,C,T,H,W] view): pass 1 writes per-slice
//     (mean, M2) partials, pass 2 merges them (Chan) and normalises.
#include "common.cuh"
#include "ptx.cuh"

namespace mvoc {

constexpr int GN_THREADS = 512;
constexpr int GN_MAX_SPLIT = 64;
constexpr int64_t GN_SMEM_SLAB_MAX = 200 * 1024;

__device__ __forceinline__ float block_sum(float v, float* red /*[32]*/) {
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    __syncthreads();  // protect `red` from the previous use
    if (lane == 0) red[w] = v;
    __syncthreads();
    float t = (lane < (blockDim.x >> 5)) ? red[lane] : 0.0f;
    t = warp_sum(t);
    return t;  // every thread holds the total
}

// ---------------------------------------------------------------- path A ---
template <typename T>
__global__ void __launch_bounds__(GN_THREADS) gn_slab_kernel(
    const T* x, T* y, const T* __restrict__ gamma,
    const T* __restrict__ beta, int C, int64_t S, int G, float eps, int silu) {
    extern __shared__ __align__(128) uint8_t gn_smem[];
    __shared__ float red[32];
    __shared__ __align__(8) uint64_t bar;
    const int Cg = C / G;
    const int64_t slab = (int64_t)Cg * S;  // elements, multiple of 8
    const int n = blockIdx.x / G, g = blockIdx.x % G;
    const int64_t base = ((int64_t)n * C + (int64_t)g * Cg) * S;
    const uint32_t bar_a = smem_u32(&bar);
    const uint32_t buf_a = smem_u32(gn_smem);
    const uint32_t bytes = (uint32_t)(slab * sizeof(T));
    constexpr uint32_t CHUNK = 16 * 1024;

    if (threadIdx.x == 0) {
        ptx::mbar_init(bar_a, 1);
        ptx::fence_mbar_init();
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        if (threadIdx.x == 0) ptx::mbar_expect_tx(bar_a, bytes);
        __syncwarp();
        for (uint32_t off = threadIdx.x * CHUNK; off < bytes; off += 32 * CHUNK) {
            const uint32_t sz = min(CHUNK, bytes - off);
            ptx::bulk_load(buf_a + off, reinterpret_cast<const uint8_t*>(x + base) + off, sz, bar_a);
        }
    }
    ptx::mbar_wait(bar_a, 0, 100);

    Vec16* sv = reinterpret_cast<Vec16*>(gn_smem);
    const int64_t nvec = slab >> 3;
    float s = 0.0f;
    for (int64_t i = threadIdx.x; i < nvec; i += GN_THREADS) {
        float f[8];
        unpack8<T>(sv[i], f);
#pragma unroll
        for (int e = 0; e < 8; ++e) s += f[e];
    }
    const float mean = block_sum(s, red) / (float)slab;
    float q = 0.0f;
    for (int64_t i = threadIdx.x; i < nvec; i += GN_THREADS) {
        float f[8];
        unpack8<T>(sv[i], f);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const float d = f[e] - mean;
            q += d * d;
        }
    }
    const float var = block_sum(q, red) / (float)slab;
    const float rstd = rsqrtf(var + eps);
    const int64_t vec_per_ch = S >> 3;
    for (int64_t i = threadIdx.x; i < nvec; i += GN_THREADS) {
        const int c = g * Cg + (int)(i / vec_per_ch);
        const float ga = Elem<T>::to_f(gamma[c]) * rstd;
        const float be = Elem<T>::to_f(beta[c]) - mean * ga;
        float f[8];
        unpack8<T>(sv[i], f);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            float v = f[e] * ga + be;
            f[e] = silu ? silu_f(v) : v;
        }
        sv[i] = pack8<T>(f);
    }
    ptx::fence_proxy_async_smem();
    __syncthreads();
    if (threadIdx.x < 32) {
        for (uint32_t off = threadIdx.x * CHUNK; off < bytes; off += 32 * CHUNK) {
            const uint32_t sz = min(CHUNK, bytes - off);
            ptx::bulk_store(reinterpret_cast<uint8_t*>(y + base) + off, buf_a + off, sz);
        }
        ptx::bulk_commit();
        ptx::bulk_wait_read0();
    }
}

// ---------------------------------------------------------------- path B ---
struct GNSplit {
    int64_t seg;          // elements in one (n, group) segment = Cg*S
    int64_t slice;        // elements per slice (multiple of V)
    int split;            // slices per segment
};

// partial[(n*G+g)*split + s] = (mean, M2) of that slice
template <typename T, int V>
__global__ void __launch_bounds__(256) gn_stats_kernel(const T* __restrict__ x,
                                                      float2* __restrict__ partial, int C,
                                                      int64_t S, int G, GNSplit sp) {
    __shared__ float red[32];
    const int seg_id = blockIdx.y;  // n*G + g
    const int n = seg_id / G, g = seg_id % G;
    const int Cg = C / G;
    const int64_t base = ((int64_t)n * C + (int64_t)g * Cg) * S;
    const int64_t lo = (int64_t)blockIdx.x * sp.slice;
    const int64_t hi = min(sp.seg, lo + sp.slice);
    const int64_t cnt = hi - lo;
    if (cnt <= 0) {
        if (threadIdx.x == 0) partial[(int64_t)seg_id * sp.split + blockIdx.x] = make_float2(0.f, 0.f);
        return;
    }
    const T* p = x + base + lo;
    const float shift = Elem<T>::to_f(p[0]);
    float s1 = 0.0f, s2 = 0.0f;
    if (V == 8) {
        const int64_t nvec = cnt >> 3;
        for (int64_t i = threadIdx.x; i < nvec; i += 256) {
            float f[8];
            unpack8<T>(ld_global16(p + (i << 3)), f);
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const float d = f[e] - shift;
                s1 += d;
                s2 += d * d;
            }
        }
    } else {
        for (int64_t i = threadIdx.x; i < cnt; i += 256) {
            const float d = Elem<T>::to_f(p[i]) - shift;
            s1 += d;
            s2 += d * d;
        }
    }
    s1 = block_sum(s1, red);
    s2 = block_sum(s2, red);
    if (threadIdx.x == 0) {
        const float m = s1 / (float)cnt;
        partial[(int64_t)seg_id * sp.split + blockIdx.x] =
            make_float2(shift + m, fmaxf(s2 - s1 * m, 0.0f));
    }
}

__device__ __forceinline__ void chan_merge(float& na, float& ma, float& qa, float nb, float mb,
                                           float qb) {
    if (nb == 0.0f) return;
    const float nt = na + nb;
    const float d = mb - ma;
    ma += d * (nb / nt);
    qa += qb + d * d * (na * nb / nt);
    na = nt;
}

template <typename T, int V>
__global__ void __launch_bounds__(256) gn_apply_kernel(
    const T* x, T* y, const T* __restrict__ gamma,
    const T* __restrict__ beta, const float2* __restrict__ partial, int C, int64_t S, int G,
    int frames, float eps, int silu, GNSplit sp) {
    __shared__ float s_mean, s_rstd;
    const int seg_id = blockIdx.y;
    const int n = seg_id / G, g = seg_id % G;
    const int Cg = C / G;
    if (threadIdx.x < 32) {
        // merge the partials of all `frames` segments that share statistics
        const int n0 = (n / frames) * frames;
        const int total = frames * sp.split;
        float na = 0.f, ma = 0.f, qa = 0.f;
        for (int i = threadIdx.x; i < total; i += 32) {
            const int fr = i / sp.split, s = i % sp.split;
            const float2 pm = partial[((int64_t)(n0 + fr) * G + g) * sp.split + s];
            const int64_t lo = (int64_t)s * sp.slice;
            const float cnt = (float)max((int64_t)0, min(sp.seg, lo + sp.slice) - lo);
            chan_merge(na, ma, qa, cnt, pm.x, pm.y);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float nb = __shfl_xor_sync(0xffffffffu, na, o);
            const float mb = __shfl_xor_sync(0xffffffffu, ma, o);
            const float qb = __shfl_xor_sync(0xffffffffu, qa, o);
            chan_merge(na, ma, qa, nb, mb, qb);
        }
        if (threadIdx.x == 0) {
            s_mean = ma;
            s_rstd = rsqrtf(qa / na + eps);
        }
    }
    __syncthreads();
    const float mean = s_mean, rstd = s_rstd;
    const int64_t base = ((int64_t)n * C + (int64_t)g * Cg) * S;
    const int64_t lo = (int64_t)blockIdx.x * sp.slice;
    const int64_t hi = min(sp.seg, lo + sp.slice);
    if (V == 8) {
        const int64_t vec_per_ch = S >> 3;
        for (int64_t i = (lo >> 3) + threadIdx.x; i < (hi >> 3); i += 256) {
            const int c = g * Cg + (int)(i / vec_per_ch);
            const float ga = Elem<T>::to_f(gamma[c]) * rstd;
            const float be = Elem<T>::to_f(beta[c]) - mean * ga;
            float f[8];
            unpack8<T>(ld_stream16(x + base + (i << 3)), f);
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const float v = f[e] * ga + be;
                f[e] = silu ? silu_f(v) : v;
            }
            st_stream16(y + base + (i << 3), pack8<T>(f));
        }
    } else {
        for (int64_t i = lo + threadIdx.x; i < hi; i += 256) {
            const int c = g * Cg + (int)(i / S);
            const float ga = Elem<T>::to_f(gamma[c]) * rstd;
            const float be = Elem<T>::to_f(beta[c]) - mean * ga;
            const float v = Elem<T>::to_f(x[base + i]) * ga + be;
            y[base + i] = Elem<T>::from_f(silu ? silu_f(v) : v);
        }
    }
}

template <typename T>
static int gn_launch(const void* x, void* y, const void* gamma, const void* beta, int64_t N, int C,
                     int64_t S, int G, int frames, float eps, int silu, void* ws, cudaStream_t st) {
    const T* xp = reinterpret_cast<const T*>(x);
    T* yp = reinterpret_cast<T*>(y);
    const T* gp = reinterpret_cast<const T*>(gamma);
    const T* bp = reinterpret_cast<const T*>(beta);
    const int Cg = C / G;
    const int64_t seg = (int64_t)Cg * S;
    const bool vec = (S % 8 == 0) && ((uintptr_t)x % 16 == 0) && ((uintptr_t)y % 16 == 0);
    const int64_t slab_bytes = seg * (int64_t)sizeof(T);
    if (frames == 1 && vec && slab_bytes <= GN_SMEM_SLAB_MAX && sizeof(T) == 2) {
        static bool smem_set[64] = {false};
        const int rc = set_max_dynamic_smem((const void*)gn_slab_kernel<T>, (int)GN_SMEM_SLAB_MAX, smem_set,
                                            "mvoc_groupnorm_silu");
        if (rc != MVOC_OK) return rc;
        gn_slab_kernel<T><<<(unsigned)(N * G), GN_THREADS, (size_t)slab_bytes, st>>>(
            xp, yp, gp, bp, C, S, G, eps, silu);
        return check_launch("mvoc_groupnorm_silu(slab)");
    }
    GNSplit sp;
    sp.seg = seg;
    int split = (int)((slab_bytes + 32 * 1024 - 1) / (32 * 1024));
    split = split < 1 ? 1 : (split > GN_MAX_SPLIT ? GN_MAX_SPLIT : split);
    int64_t slice = (seg + split - 1) / split;
    if (vec) slice = (slice + 7) & ~(int64_t)7;
    sp.slice = slice;
    sp.split = split;
    float2* part = reinterpret_cast<float2*>(ws);
    dim3 grid(split, (unsigned)(N * G));
    if (vec) {
        gn_stats_kernel<T, 8><<<grid, 256, 0, st>>>(xp, part, C, S, G, sp);
        gn_apply_kernel<T, 8><<<grid, 256, 0, st>>>(xp, yp, gp, bp, part, C, S, G, frames, eps, silu, sp);
    } else {
        gn_stats_kernel<T, 1><<<grid, 256, 0, st>>>(xp, part, C, S, G, sp);
        gn_apply_kernel<T, 1><<<grid, 256, 0, st>>>(xp, yp, gp, bp, part, C, S, G, frames, eps, silu, sp);
    }
    return check_launch("mvoc_groupnorm_silu(split)");
}

}  // namespace mvoc

using namespace mvoc;

extern "C" int64_t mvoc_groupnorm_workspace_bytes(int64_t N, int G) {
    return N * (int64_t)G * GN_MAX_SPLIT * (int64_t)sizeof(float2);
}

extern "C" int mvoc_groupnorm_silu(const void* x, void* y, const void* gamma, const void* beta,
                                   int64_t N, int C, int64_t S, int G, int frames_per_stat,
                                   float eps, int silu, int dtype, void* workspace, void* stream) {
    MVOC_REQUIRE(x && y && gamma && beta && workspace, MVOC_ERR_INVALID_ARG,
                 "mvoc_groupnorm_silu: null pointer");
    MVOC_REQUIRE(N > 0 && C > 0 && S > 0 && G > 0 && C % G == 0, MVOC_ERR_INVALID_ARG,
                 "mvoc_groupnorm_silu: bad shape N=%lld C=%d S=%lld G=%d", (long long)N, C,
                 (long long)S, G);
    MVOC_REQUIRE(frames_per_stat >= 1 && N % frames_per_stat == 0, MVOC_ERR_INVALID_ARG,
                 "mvoc_groupnorm_silu: N=%lld not a multiple of frames_per_stat=%d", (long long)N,
                 frames_per_stat);
    MVOC_REQUIRE(N * G < 65536, MVOC_ERR_UNSUPPORTED,
                 "mvoc_groupnorm_silu: N*G=%lld exceeds grid.y limit", (long long)(N * G));
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == MVOC_BF16)
        return gn_launch<__nv_bfloat16>(x, y, gamma, beta, N, C, S, G, frames_per_stat, eps, silu,
                                        workspace, st);
    if (dtype == MVOC_F16)
        return gn_launch<__half>(x, y, gamma, beta, N, C, S, G, frames_per_stat, eps, silu,
                                 workspace, st);
    set_error("mvoc_groupnorm_silu: dtype %d unsupported (bf16/f16 only)", dtype);
    return MVOC_ERR_UNSUPPORTED;
}
