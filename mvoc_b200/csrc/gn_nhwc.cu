// GroupNorm (+SiLU, + fused per-(frame, channel) add) for channels-last activations [N, S, C], and
// the fused GEGLU gate — the HBM-bound normalisation / activation kernels of the NHWC host path.
//
// Reference call sites: i2vgen-xl/pnp_utils.py:909-910 and :941-965 (resnet norm1, `+ temb`, norm2 + SiLU),
// :1048-1051 (TemporalConvLayer GN->SiLU heads, statistics over the [B,C,T,H,W] view), :430 and :185-188
// (transformer norms), pipelines/pipeline_i2vgen_xl.py:351-352 (conv_norm_out + SiLU); GEGLU is
// `ff.net.0` of BasicTransformerBlock (pnp_utils.py:335; diffusers GEGLU: proj -> x * gelu(gate)).
//
// Channels-last makes every 1x1 conv / Linear / LayerNorm a plain row-wise op and removes the
// NCHW<->NLC permutes (pnp_utils.py:434, :502, :189, :207-213).  GroupNorm then reduces over
// (tokens x C/G channels): three launches
//   stats    : per (n, chunk of tokens) per-group (mean, M2), shifted sums in fp32          [read  X]
//   finalize : Chan-merge of the partials of one statistics group (T frames, all chunks,
//              and — for multi-GPU pixel shards — the partial sets gathered from all ranks)   [tiny]
//   apply    : y = silu?((x + add - mean) * rstd * gamma + beta), 128-bit accesses         [read X, write Y]
// `add` is the resnet time embedding: GN(conv1(h) + temb) without a separate pass over the tensor.
#include "common.cuh"

namespace mvoc {

constexpr int GNH_MAX_CHUNKS = 64;

struct GNHParams {
    const void* x;
    void* y;
    const void* gamma;
    const void* beta;
    const void* add;        // [N, C] or null
    float2* partial;        // [N, G, chunks] (mean, M2)
    const float2* stat;     // [N / frames, G] (mean, rstd) — apply only
    int64_t S;
    int C, G, chunks;
    int64_t tokens_per_chunk;
    int R;                  // token lanes per CTA; blockDim = (C/8) * R
    int frames;             // statistics shared by `frames` consecutive n
    float eps;
    int silu;
};

template <typename T>
__global__ void gnh_stats_kernel(GNHParams p) {
    // smem: part1[R][C], part2[R][C] (per-lane partial sums, reduced in a fixed order => deterministic),
    //       s1[C], s2[C], shift[C]
    extern __shared__ float gnh_smem[];
    const int C = p.C, VC = C >> 3, Cg = C / p.G, R = p.R;
    float* part1 = gnh_smem;
    float* part2 = part1 + (size_t)R * C;
    float* s1 = part2 + (size_t)R * C;
    float* s2 = s1 + C;
    float* sh = s2 + C;
    const int n = blockIdx.y, chunk = blockIdx.x;
    const int vc = threadIdx.x % VC, r = threadIdx.x / VC;
    const int64_t t0 = (int64_t)chunk * p.tokens_per_chunk;
    const int64_t t1 = min(p.S, t0 + p.tokens_per_chunk);
    const T* xb = reinterpret_cast<const T*>(p.x) + (int64_t)n * p.S * C + vc * 8;
    float addv[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) addv[e] = 0.0f;
    if (p.add) unpack8<T>(ld_global16(reinterpret_cast<const T*>(p.add) + (int64_t)n * C + vc * 8), addv);
    float shift[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) shift[e] = 0.0f;
    if (t0 < t1) {  // common per-channel shift (first token of the chunk) against cancellation
        unpack8<T>(ld_global16(xb + t0 * C), shift);
#pragma unroll
        for (int e = 0; e < 8; ++e) shift[e] += addv[e];
    }
    float a1[8], a2[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) a1[e] = a2[e] = 0.0f;
    int64_t t = t0 + r;
    // four independent 16-byte loads in flight per thread
    for (; t + 3 * R < t1; t += 4 * R) {
        Vec16 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = ld_stream16(xb + (t + u * R) * C);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            float f[8];
            unpack8<T>(v[u], f);
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const float d = f[e] + addv[e] - shift[e];
                a1[e] += d;
                a2[e] += d * d;
            }
        }
    }
    for (; t < t1; t += R) {
        float f[8];
        unpack8<T>(ld_stream16(xb + t * C), f);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const float d = f[e] + addv[e] - shift[e];
            a1[e] += d;
            a2[e] += d * d;
        }
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        part1[(size_t)r * C + vc * 8 + e] = a1[e];
        part2[(size_t)r * C + vc * 8 + e] = a2[e];
    }
    if (r == 0) {
#pragma unroll
        for (int e = 0; e < 8; ++e) sh[vc * 8 + e] = shift[e];
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float x1 = 0.0f, x2 = 0.0f;
        for (int rr = 0; rr < R; ++rr) {
            x1 += part1[(size_t)rr * C + c];
            x2 += part2[(size_t)rr * C + c];
        }
        s1[c] = x1;
        s2[c] = x2;
    }
    __syncthreads();
    // one thread per group: Chan-merge the per-channel statistics of its C/G channels
    if (threadIdx.x < p.G) {
        const int g = threadIdx.x;
        const float cnt = (float)(t1 > t0 ? (t1 - t0) : 0);
        float na = 0.f, ma = 0.f, qa = 0.f;
        if (cnt > 0.f) {
            for (int c = g * Cg; c < (g + 1) * Cg; ++c) {
                const float m = s1[c] / cnt;
                const float mb = sh[c] + m;
                const float qb = fmaxf(s2[c] - s1[c] * m, 0.0f);
                const float nt = na + cnt;
                const float d = mb - ma;
                ma += d * (cnt / nt);
                qa += qb + d * d * (na * cnt / nt);
                na = nt;
            }
        }
        p.partial[((int64_t)n * p.G + g) * p.chunks + chunk] = make_float2(ma, qa);
    }
}

// One warp per (statistics group, g): merge frames x chunks x sets partials.
// partial sets are laid out [set][N][G][chunks]; counts[set*chunks + chunk] tokens*Cg elements each.
__global__ void gnh_finalize_kernel(const float2* __restrict__ partial, float2* __restrict__ stat,
                                    const float* __restrict__ counts, int N, int G, int chunks,
                                    int frames, int sets, float eps) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    const int n_groups = (N / frames) * G;
    if (warp >= n_groups) return;
    const int sg = warp / G, g = warp % G;
    const int per_set = frames * chunks;
    const int total = per_set * sets;
    float na = 0.f, ma = 0.f, qa = 0.f;
    for (int i = lane; i < total; i += 32) {
        const int set = i / per_set, rem = i % per_set;
        const int fr = rem / chunks, ch = rem % chunks;
        const float2 pm = partial[(((int64_t)set * N + (sg * frames + fr)) * G + g) * chunks + ch];
        const float nb = counts[set * chunks + ch];
        if (nb > 0.f) {
            const float nt = na + nb;
            const float d = pm.x - ma;
            ma += d * (nb / nt);
            qa += pm.y + d * d * (na * nb / nt);
            na = nt;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float nb = __shfl_xor_sync(0xffffffffu, na, o);
        const float mb = __shfl_xor_sync(0xffffffffu, ma, o);
        const float qb = __shfl_xor_sync(0xffffffffu, qa, o);
        if (nb > 0.f) {
            const float nt = na + nb;
            const float d = mb - ma;
            ma += d * (nb / nt);
            qa += qb + d * d * (na * nb / nt);
            na = nt;
        }
    }
    if (lane == 0) stat[warp] = make_float2(ma, rsqrtf(qa / fmaxf(na, 1.0f) + eps));
}

template <typename T>
__global__ void gnh_apply_kernel(GNHParams p) {
    const int C = p.C, VC = C >> 3, Cg = C / p.G;
    const int n = blockIdx.y, chunk = blockIdx.x;
    const int vc = threadIdx.x % VC, r = threadIdx.x / VC;
    const int64_t t0 = (int64_t)chunk * p.tokens_per_chunk;
    const int64_t t1 = min(p.S, t0 + p.tokens_per_chunk);
    const T* xb = reinterpret_cast<const T*>(p.x) + (int64_t)n * p.S * C + vc * 8;
    T* yb = reinterpret_cast<T*>(p.y) + (int64_t)n * p.S * C + vc * 8;
    float ga[8], be[8], sc[8], sf[8];
    unpack8<T>(ld_global16(reinterpret_cast<const T*>(p.gamma) + vc * 8), ga);
    unpack8<T>(ld_global16(reinterpret_cast<const T*>(p.beta) + vc * 8), be);
    float addv[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) addv[e] = 0.0f;
    if (p.add) unpack8<T>(ld_global16(reinterpret_cast<const T*>(p.add) + (int64_t)n * C + vc * 8), addv);
    const float2* st = p.stat + (int64_t)(n / p.frames) * p.G;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        const float2 ms = st[(vc * 8 + e) / Cg];
        sc[e] = ga[e] * ms.y;
        sf[e] = be[e] + (addv[e] - ms.x) * sc[e];
    }
    const int R = p.R;
    int64_t t = t0 + r;
    for (; t + 3 * R < t1; t += 4 * R) {  // four independent 16-byte loads in flight per thread
        Vec16 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = ld_stream16(xb + (t + u * R) * C);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            float f[8];
            unpack8<T>(v[u], f);
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const float w = f[e] * sc[e] + sf[e];
                f[e] = p.silu ? silu_f(w) : w;
            }
            st_stream16(yb + (t + u * R) * C, pack8<T>(f));
        }
    }
    for (; t < t1; t += R) {
        float f[8];
        unpack8<T>(ld_stream16(xb + t * C), f);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const float w = f[e] * sc[e] + sf[e];
            f[e] = p.silu ? silu_f(w) : w;
        }
        st_stream16(yb + t * C, pack8<T>(f));
    }
}

static void gnh_geometry(int64_t S, int C, int esize, int* chunks, int64_t* tpc, int* R) {
    const int VC = C / 8;
    int r = 320 / VC;
    if (r < 1) r = 1;
    if (r > 32) r = 32;
    while (VC * r > 1024) --r;
    int64_t ch = (S * (int64_t)C * esize + 160 * 1024 - 1) / (160 * 1024);
    if (ch < 1) ch = 1;
    if (ch > GNH_MAX_CHUNKS) ch = GNH_MAX_CHUNKS;
    int64_t t = (S + ch - 1) / ch;
    *chunks = (int)((S + t - 1) / t);
    *tpc = t;
    *R = r;
}

// y[m, j] = x[m, j] * gelu(x[m, F + j]); exact (erf) GELU as in torch.nn.functional.gelu
template <typename T>
__global__ void __launch_bounds__(256) geglu_kernel(const T* __restrict__ x, T* __restrict__ y, int64_t M,
                                                    int F) {
    const int vf = F >> 3;
    const int64_t items = M * vf;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t it = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; it < items; it += stride) {
        const int64_t m = it / vf;
        const int j = (int)(it - m * vf) << 3;
        float a[8], g[8];
        unpack8<T>(ld_stream16(x + m * 2 * F + j), a);
        unpack8<T>(ld_stream16(x + m * 2 * F + F + j), g);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const float ge = 0.5f * g[e] * (1.0f + erff(g[e] * 0.70710678118654752f));
            a[e] = a[e] * ge;  // one rounding at the store (the reference rounds gelu(gate) first)
        }
        st_stream16(y + it * 8, pack8<T>(a));
    }
}

}  // namespace mvoc

using namespace mvoc;

extern "C" int64_t mvoc_groupnorm_nhwc_partial_count(int64_t N, int G) {
    return N * (int64_t)G * GNH_MAX_CHUNKS;
}

extern "C" int mvoc_groupnorm_nhwc_geometry(int64_t S, int C, int dtype, int* chunks,
                                            int64_t* tokens_per_chunk) {
    MVOC_REQUIRE(S > 0 && C > 0 && C % 8 == 0, MVOC_ERR_UNSUPPORTED,
                 "mvoc_groupnorm_nhwc_geometry: need S>0 and C%%8==0 (S=%lld C=%d)", (long long)S, C);
    int R;
    gnh_geometry(S, C, dtype == MVOC_F32 ? 4 : 2, chunks, tokens_per_chunk, &R);
    return MVOC_OK;
}

static int gnh_check(const char* name, int64_t N, int64_t S, int C, int G, int frames, int dtype) {
    MVOC_REQUIRE(N > 0 && S > 0 && C > 0 && G > 0 && C % G == 0, MVOC_ERR_INVALID_ARG,
                 "%s: bad shape N=%lld S=%lld C=%d G=%d", name, (long long)N, (long long)S, C, G);
    MVOC_REQUIRE(C % 8 == 0 && C / 8 <= 1024, MVOC_ERR_UNSUPPORTED, "%s: C=%d must be a multiple of 8 (<= 8192)", name, C);
    MVOC_REQUIRE(G <= 32 * 4, MVOC_ERR_UNSUPPORTED, "%s: G=%d too large", name, G);
    MVOC_REQUIRE(frames >= 1 && N % frames == 0, MVOC_ERR_INVALID_ARG,
                 "%s: N=%lld not a multiple of frames_per_stat=%d", name, (long long)N, frames);
    MVOC_REQUIRE(N < 65536, MVOC_ERR_UNSUPPORTED, "%s: N=%lld exceeds grid.y", name, (long long)N);
    MVOC_REQUIRE(dtype == MVOC_BF16 || dtype == MVOC_F16, MVOC_ERR_UNSUPPORTED,
                 "%s: dtype %d unsupported (bf16/f16 only)", name, dtype);
    return MVOC_OK;
}

extern "C" int mvoc_groupnorm_nhwc_stats(const void* x, const void* add, void* partial, int64_t N,
                                         int64_t S, int C, int G, int dtype, void* stream) {
    MVOC_REQUIRE(x && partial, MVOC_ERR_INVALID_ARG, "mvoc_groupnorm_nhwc_stats: null pointer");
    int rc = gnh_check("mvoc_groupnorm_nhwc_stats", N, S, C, G, 1, dtype);
    if (rc != MVOC_OK) return rc;
    GNHParams p{};
    p.x = x;
    p.add = add;
    p.partial = reinterpret_cast<float2*>(partial);
    p.S = S;
    p.C = C;
    p.G = G;
    gnh_geometry(S, C, 2, &p.chunks, &p.tokens_per_chunk, &p.R);
    const int threads = (C / 8) * p.R;
    MVOC_REQUIRE(threads >= G, MVOC_ERR_UNSUPPORTED, "mvoc_groupnorm_nhwc_stats: C=%d too small for G=%d", C, G);
    dim3 grid(p.chunks, (unsigned)N);
    const size_t smem = (2 * (size_t)p.R + 3) * (size_t)C * sizeof(float);
    MVOC_REQUIRE(smem <= 96 * 1024, MVOC_ERR_UNSUPPORTED, "mvoc_groupnorm_nhwc_stats: C=%d needs %zu B of smem", C, smem);
    static bool smem_set[2][64] = {};
    const bool bf16 = dtype == MVOC_BF16;
    const void* kernel = bf16 ? (const void*)gnh_stats_kernel<__nv_bfloat16> : (const void*)gnh_stats_kernel<__half>;
    if ((rc = set_max_dynamic_smem(kernel, 96 * 1024, smem_set[bf16], "mvoc_groupnorm_nhwc_stats")) != MVOC_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (bf16) gnh_stats_kernel<__nv_bfloat16><<<grid, threads, smem, st>>>(p);
    else gnh_stats_kernel<__half><<<grid, threads, smem, st>>>(p);
    return check_launch("mvoc_groupnorm_nhwc_stats");
}

extern "C" int mvoc_groupnorm_nhwc_finalize(const void* partial, const void* counts, void* stat,
                                            int64_t N, int G, int chunks, int frames_per_stat, int sets,
                                            float eps, void* stream) {
    MVOC_REQUIRE(partial && counts && stat, MVOC_ERR_INVALID_ARG, "mvoc_groupnorm_nhwc_finalize: null pointer");
    MVOC_REQUIRE(N > 0 && G > 0 && chunks > 0 && sets > 0 && frames_per_stat > 0 && N % frames_per_stat == 0,
                 MVOC_ERR_INVALID_ARG, "mvoc_groupnorm_nhwc_finalize: bad arguments");
    const int n_groups = (int)(N / frames_per_stat) * G;
    const int threads = 128;
    const int grid = (n_groups * 32 + threads - 1) / threads;
    gnh_finalize_kernel<<<grid, threads, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const float2*>(partial), reinterpret_cast<float2*>(stat),
        reinterpret_cast<const float*>(counts), (int)N, G, chunks, frames_per_stat, sets, eps);
    return check_launch("mvoc_groupnorm_nhwc_finalize");
}

extern "C" int mvoc_groupnorm_nhwc_apply(const void* x, void* y, const void* gamma, const void* beta,
                                         const void* add, const void* stat, int64_t N, int64_t S, int C,
                                         int G, int frames_per_stat, int silu, int dtype, void* stream) {
    MVOC_REQUIRE(x && y && gamma && beta && stat, MVOC_ERR_INVALID_ARG, "mvoc_groupnorm_nhwc_apply: null pointer");
    int rc = gnh_check("mvoc_groupnorm_nhwc_apply", N, S, C, G, frames_per_stat, dtype);
    if (rc != MVOC_OK) return rc;
    GNHParams p{};
    p.x = x;
    p.y = y;
    p.gamma = gamma;
    p.beta = beta;
    p.add = add;
    p.stat = reinterpret_cast<const float2*>(stat);
    p.S = S;
    p.C = C;
    p.G = G;
    p.frames = frames_per_stat;
    p.silu = silu;
    gnh_geometry(S, C, 2, &p.chunks, &p.tokens_per_chunk, &p.R);
    const int threads = (C / 8) * p.R;
    dim3 grid(p.chunks, (unsigned)N);
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == MVOC_BF16) gnh_apply_kernel<__nv_bfloat16><<<grid, threads, 0, st>>>(p);
    else gnh_apply_kernel<__half><<<grid, threads, 0, st>>>(p);
    return check_launch("mvoc_groupnorm_nhwc_apply");
}

extern "C" int mvoc_geglu(const void* x, void* y, int64_t M, int F, int dtype, void* stream) {
    MVOC_REQUIRE(x && y, MVOC_ERR_INVALID_ARG, "mvoc_geglu: null pointer");
    MVOC_REQUIRE(M >= 0 && F > 0 && F % 8 == 0, MVOC_ERR_UNSUPPORTED, "mvoc_geglu: F=%d must be a positive multiple of 8", F);
    MVOC_REQUIRE(dtype == MVOC_BF16 || dtype == MVOC_F16, MVOC_ERR_UNSUPPORTED, "mvoc_geglu: dtype %d unsupported", dtype);
    MVOC_REQUIRE(((uintptr_t)x % 16 == 0) && ((uintptr_t)y % 16 == 0), MVOC_ERR_INVALID_ARG, "mvoc_geglu: pointers must be 16-byte aligned");
    if (M == 0) return MVOC_OK;
    const int64_t items = M * (F / 8);
    int64_t want = (items + 255) / 256;
    const int64_t cap = (int64_t)num_sms() * 16;
    const int grid = (int)(want < cap ? want : cap);
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == MVOC_BF16)
        geglu_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>((const __nv_bfloat16*)x, (__nv_bfloat16*)y, M, F);
    else
        geglu_kernel<__half><<<grid, 256, 0, st>>>((const __half*)x, (__half*)y, M, F);
    return check_launch("mvoc_geglu");
}
