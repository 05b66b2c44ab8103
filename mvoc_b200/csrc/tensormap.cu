// TMA tensor maps of the tensor-core kernels (attn_tc, attn_wide, gemm_tc): one stride rule, one driver lookup.
#include "common.cuh"

namespace mvoc {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
        if (e == cudaSuccess && qres == cudaDriverEntryPointSuccess) fn = (EncodeTiledFn)p;
    }
    return fn;
}

// TMA cannot broadcast: a zero stride along a dimension of extent > 1 would make the map read past the tensor.
int check_map4(const int64_t (&dims)[4], const int64_t (&str)[3], const char* what, const char* operand) {
    for (int i = 0; i < 3; ++i)
        MVOC_REQUIRE(dims[i + 1] == 1 || (str[i] > 0 && str[i] % 8 == 0), MVOC_ERR_UNSUPPORTED,
                     "%s: %s stride %lld of dimension %d (extent %lld) is not a positive multiple of 8 elements", what,
                     operand, (long long)str[i], i + 1, (long long)dims[i + 1]);
    return MVOC_OK;
}

int make_map4(CUtensorMap* m, const void* base, int dtype, const int64_t (&dims)[4], const int64_t (&str)[3],
              const int (&box)[4], int elem_stride, CUtensorMapSwizzle swz, const char* what, const char* operand) {
    int rc = check_map4(dims, str, what, operand);
    if (rc != MVOC_OK) return rc;
    MVOC_REQUIRE(elem_stride >= 1 && elem_stride <= 8, MVOC_ERR_UNSUPPORTED, "%s: %s element stride %d (1..8)", what,
                 operand, elem_stride);
    EncodeTiledFn fn = get_encode_fn();
    MVOC_REQUIRE(fn != nullptr, MVOC_ERR_DRIVER, "%s: cuTensorMapEncodeTiled unavailable", what);
    cuuint64_t d[4], s[3];
    cuuint32_t b[4], estr[4] = {1, (cuuint32_t)elem_stride, (cuuint32_t)elem_stride, 1};
    for (int i = 0; i < 4; ++i) d[i] = (cuuint64_t)dims[i], b[i] = (cuuint32_t)box[i];
    for (int i = 0; i < 3; ++i)   // bytes; an extent-1 dimension is never stepped, so it gets the packed stride
        s[i] = dims[i + 1] == 1 ? (i == 0 ? d[0] * 2 : s[i - 1] * d[i]) : (cuuint64_t)str[i] * 2;
    CUresult r = fn(m, dtype == MVOC_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4,
                    const_cast<void*>(base), d, s, b, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    MVOC_REQUIRE(r == CUDA_SUCCESS, MVOC_ERR_DRIVER,
                 "%s: cuTensorMapEncodeTiled(%s) failed with CUresult %d (dims %lld,%lld,%lld,%lld strides "
                 "%lld,%lld,%lld box %d,%d,%d,%d element stride %d)",
                 what, operand, (int)r, (long long)dims[0], (long long)dims[1], (long long)dims[2], (long long)dims[3],
                 (long long)str[0], (long long)str[1], (long long)str[2], box[0], box[1], box[2], box[3], elem_stride);
    return MVOC_OK;
}

}  // namespace mvoc
