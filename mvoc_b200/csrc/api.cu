// Library-level entry points: version, error text, device check.
#include <stdarg.h>
#include <string.h>
#include "common.cuh"

namespace mvoc {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: CUDA error %d (%s)", what, (int)e, cudaGetErrorString(e));
        return MVOC_ERR_CUDA;
    }
    return MVOC_OK;
}

int set_max_dynamic_smem(const void* kernel, int bytes, bool (&done)[64], const char* what) {
    int dev = 0;
    cudaGetDevice(&dev);
    const bool tracked = dev >= 0 && dev < 64;
    if (tracked && done[dev]) return MVOC_OK;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    MVOC_REQUIRE(e == cudaSuccess, MVOC_ERR_CUDA, "%s: cudaFuncSetAttribute: %s", what, cudaGetErrorString(e));
    if (tracked) done[dev] = true;
    return MVOC_OK;
}

}  // namespace mvoc

extern "C" const char* mvoc_version(void) { return "mvoc_b200 0.1.0 (sm_100a)"; }

extern "C" const char* mvoc_last_error(void) { return mvoc::g_err; }

extern "C" int mvoc_device_check(int device) {
    cudaDeviceProp prop;
    cudaError_t e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) {
        mvoc::set_error("mvoc_device_check: cudaGetDeviceProperties(%d) failed: %s", device,
                        cudaGetErrorString(e));
        return MVOC_ERR_CUDA;
    }
    if (prop.major != 10) {
        mvoc::set_error("mvoc_device_check: device %d is sm_%d%d; this library is sm_100a only",
                        device, prop.major, prop.minor);
        return MVOC_ERR_UNSUPPORTED;
    }
    return MVOC_OK;
}
