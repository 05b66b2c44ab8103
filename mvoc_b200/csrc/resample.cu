// Nearest-neighbour 2x upsampling of a channels-last activation [N, H, W, C] -> [N, 2H, 2W, C]: the
// `F.interpolate(scale_factor=2.0, mode="nearest")` of diffusers' Upsample2D inside the up blocks (un-vendored
// dependency; reached from i2vgen-xl/pipelines/pipeline_i2vgen_xl.py:318-350 through UpBlock3D / CrossAttnUpBlock3D,
// `upsample_size` at :328-329).  HBM-bound: one read of X, one write of 4|X|.  ATen's NHWC kernel ran these three
// launches of a step at ~0.45 TB/s (1.9 ms per step, profiles/r02_launches_timed_step_summary.txt).
#include "common.cuh"

namespace mvoc {

// One thread per 16-byte vector of an INPUT pixel; it writes the vector to the four output pixels.  Consecutive
// threads walk the channels of a pixel, then the pixels of a row: reads and writes are full 128-byte lines.
__global__ void __launch_bounds__(256) upsample2x_nhwc_kernel(const uint4* __restrict__ x, uint4* __restrict__ y,
                                                              int64_t vecs, int H, int W, int VC) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t out_row = (int64_t)2 * W * VC;   // vectors per output row
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < vecs; i += stride) {
        const int64_t pix = i / VC;
        const int v = (int)(i - pix * VC);
        const int w = (int)(pix % W);
        const int64_t nh = pix / W;                 // n * H + h
        const Vec16 val = ld_stream16(x + i);
        uint4* o = y + ((nh * 2) * (int64_t)(2 * W) + 2 * w) * VC + v;
        st_stream16(o, val);
        st_stream16(o + VC, val);
        st_stream16(o + out_row, val);
        st_stream16(o + out_row + VC, val);
    }
}

// Channel concatenation of two channels-last activations: y[r, :] = [a[r, :CA], b[r, :CB]] — the
// `torch.cat([hidden_states, res_hidden_states], dim=1)` before every resnet of the up blocks (skip connections;
// un-vendored diffusers UNet3D up blocks reached from i2vgen-xl/pipelines/pipeline_i2vgen_xl.py:318-350), which
// is `dim=-1` in the channels-last layout.  A pure copy: bit-identical to torch.cat.  One thread per 16-byte
// output vector; consecutive threads write consecutive vectors of a row.
__global__ void __launch_bounds__(256) concat_lastdim_kernel(const uint4* __restrict__ a, const uint4* __restrict__ b,
                                                             uint4* __restrict__ y, int64_t vecs, int VA, int VB) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int VT = VA + VB;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < vecs; i += stride) {
        const int64_t r = i / VT;
        const int v = (int)(i - r * VT);
        const Vec16 val = v < VA ? ld_stream16(a + r * VA + v) : ld_stream16(b + r * VB + (v - VA));
        st_stream16(y + i, val);
    }
}

}  // namespace mvoc

using namespace mvoc;

extern "C" int mvoc_concat_lastdim(const void* a, const void* b, void* y, int64_t rows, int CA, int CB, int dtype,
                                   void* stream) {
    MVOC_REQUIRE(a && b && y, MVOC_ERR_INVALID_ARG, "mvoc_concat_lastdim: null pointer");
    MVOC_REQUIRE(rows >= 0 && CA > 0 && CB > 0, MVOC_ERR_INVALID_ARG,
                 "mvoc_concat_lastdim: bad shape rows=%lld CA=%d CB=%d", (long long)rows, CA, CB);
    MVOC_REQUIRE(dtype == MVOC_BF16 || dtype == MVOC_F16, MVOC_ERR_UNSUPPORTED,
                 "mvoc_concat_lastdim: dtype %d unsupported (bf16/f16 only)", dtype);
    MVOC_REQUIRE(CA % 8 == 0 && CB % 8 == 0, MVOC_ERR_UNSUPPORTED,
                 "mvoc_concat_lastdim: CA=%d and CB=%d must be multiples of 8", CA, CB);
    MVOC_REQUIRE(((uintptr_t)a % 16 == 0) && ((uintptr_t)b % 16 == 0) && ((uintptr_t)y % 16 == 0),
                 MVOC_ERR_INVALID_ARG, "mvoc_concat_lastdim: pointers must be 16-byte aligned");
    if (rows == 0) return MVOC_OK;
    const int VA = CA / 8, VB = CB / 8;
    const int64_t vecs = rows * (int64_t)(VA + VB);
    int64_t want = (vecs + 255) / 256;
    const int64_t cap = (int64_t)num_sms() * 16;
    const int grid = (int)(want < cap ? want : cap);
    concat_lastdim_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const uint4*)a, (const uint4*)b, (uint4*)y, vecs,
                                                                   VA, VB);
    return check_launch("mvoc_concat_lastdim");
}

extern "C" int mvoc_upsample_nearest2x_nhwc(const void* x, void* y, int64_t N, int H, int W, int C, int dtype,
                                            void* stream) {
    MVOC_REQUIRE(x && y, MVOC_ERR_INVALID_ARG, "mvoc_upsample_nearest2x_nhwc: null pointer");
    MVOC_REQUIRE(N >= 0 && H > 0 && W > 0 && C > 0, MVOC_ERR_INVALID_ARG,
                 "mvoc_upsample_nearest2x_nhwc: bad shape N=%lld H=%d W=%d C=%d", (long long)N, H, W, C);
    MVOC_REQUIRE(dtype == MVOC_BF16 || dtype == MVOC_F16, MVOC_ERR_UNSUPPORTED,
                 "mvoc_upsample_nearest2x_nhwc: dtype %d unsupported (bf16/f16 only)", dtype);
    MVOC_REQUIRE(C % 8 == 0, MVOC_ERR_UNSUPPORTED, "mvoc_upsample_nearest2x_nhwc: C=%d must be a multiple of 8", C);
    MVOC_REQUIRE(((uintptr_t)x % 16 == 0) && ((uintptr_t)y % 16 == 0), MVOC_ERR_INVALID_ARG,
                 "mvoc_upsample_nearest2x_nhwc: pointers must be 16-byte aligned");
    if (N == 0) return MVOC_OK;
    const int VC = C / 8;
    const int64_t vecs = N * H * (int64_t)W * VC;
    int64_t want = (vecs + 255) / 256;
    const int64_t cap = (int64_t)num_sms() * 16;
    const int grid = (int)(want < cap ? want : cap);
    upsample2x_nhwc_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const uint4*)x, (uint4*)y, vecs, H, W, VC);
    return check_launch("mvoc_upsample_nearest2x_nhwc");
}
