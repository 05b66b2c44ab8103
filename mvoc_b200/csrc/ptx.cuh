// Thin inline-PTX wrappers: mbarrier, TMA (cp.async.bulk[.tensor]), tcgen05.
// sm_100a only.  Every mbarrier wait carries a watchdog: a barrier that never
// completes traps with a message instead of hanging the GPU.
#pragma once
#include <stdint.h>
#include <stdio.h>

namespace mvoc {
namespace ptx {

// ------------------------------------------------------------- mbarrier ---
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.b32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
// Non-blocking poll: has the phase with this parity completed?  (acquire semantics like try_wait, no suspend)
__device__ __forceinline__ bool mbar_test(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.b32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
#ifndef MVOC_WATCHDOG_SPINS
#define MVOC_WATCHDOG_SPINS (1u << 24)
#endif
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int tag = 0) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins > MVOC_WATCHDOG_SPINS) {
            printf("mvoc: mbarrier watchdog: block (%d,%d,%d) thread %d tag %d parity %u\n",
                   blockIdx.x, blockIdx.y, blockIdx.z, threadIdx.x, tag, parity);
            __trap();
        }
    }
}

// ------------------------------------------------------------------ TMA ---
__device__ __forceinline__ void prefetch_tensormap(const void* tmap) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(tmap) : "memory");
}
// 4-D tiled load, coordinates innermost first.
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const void* tmap, uint32_t bar, int c0,
                                            int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes "
        "[%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(dst),
        "l"(tmap), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes,
                                          uint32_t bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
            "r"(dst),
        "l"(src), "r"(bytes), "r"(bar)
        : "memory");
}
__device__ __forceinline__ void bulk_store(void* dst, uint32_t src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() {
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void bulk_wait_read0() {
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// -------------------------------------------------------------- tcgen05 ---
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst),
                 "r"(ncols)
                 : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// mbarrier arrives once every tcgen05.mma issued so far by this thread has completed.
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
                 : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                       uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem desc]
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc,
                                       uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(d_tmem),
        "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// 32 lanes x 32 consecutive 32-bit columns: thread i of the warp owns lane
// (warp_id % 4) * 32 + i and receives columns [col, col+32).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
          "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
          "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
          "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]),
          "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]),
        "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]),
        "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]),
        "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() {
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_wait_st() {
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// Shared-memory matrix descriptor, 128-byte swizzle, sm_100 format:
// bits [0,14) addr>>4, [16,30) LBO>>4, [32,46) SBO>>4, [46,48) version=1, [61,64) layout=2.
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t addr, uint32_t lbo_bytes,
                                                    uint32_t sbo_bytes) {
    return (uint64_t)((addr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) |
           ((uint64_t)(sbo_bytes >> 4) << 32) | (1ull << 46) | (2ull << 61);
}

// Instruction descriptor for kind::f16 with fp32 accumulation and A K-major; A and B both fp16 or both bf16.
// [4,6) c=F32(1); [7,10) a, [10,13) b format (0 = fp16, 1 = bf16); 16 b_major (1 = MN-major);
// [17,23) N>>3; [24,29) M>>4.
__host__ __device__ constexpr uint32_t idesc_f16(bool fp16, int M, int N, bool b_mn_major) {
    return (1u << 4) | ((fp16 ? 0u : 1u) << 7) | ((fp16 ? 0u : 1u) << 10) | ((uint32_t)b_mn_major << 16) |
           ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// 128-byte-swizzled tiles need a 1024-byte aligned dynamic shared-memory base: trap with a message naming the
// kernel (a string literal) if `sbase` is not.
#define MVOC_REQUIRE_SMEM_1024(sbase, kernel)                                                                      \
    do {                                                                                                           \
        if (((sbase) & 1023u) != 0u) {                                                                             \
            if (threadIdx.x == 0)                                                                                  \
                printf("mvoc " kernel ": dynamic smem base 0x%x is not 1024-byte aligned\n", (sbase));             \
            __trap();                                                                                              \
        }                                                                                                          \
    } while (0)

// ---- packed fp32x2 arithmetic (sm_100: FFMA2 / FADD2 issue two fp32 ops per slot) ----------------------
__device__ __forceinline__ uint64_t pack2(float lo, float hi) {
    uint64_t v;
    asm("mov.b64 %0, {%1, %2};" : "=l"(v) : "f"(lo), "f"(hi));
    return v;
}
__device__ __forceinline__ void unpack2(uint64_t v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ uint64_t sub2(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ uint64_t mul2(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ uint64_t add2_round_down(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("add.rm.ftz.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ float max3(float a, float b, float c) {
    float d;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}

// 2^x for a pair, evaluated on the FMA pipe instead of the MUFU (which is the bottleneck of a D = 64
// softmax): Cody-Waite split x = floor(x) + f, degree-3 minimax polynomial for 2^f on [0,1) (max rel. error
// ~9e-5, invisible after the bf16 rounding of P), integer part added to the exponent field.  The technique
// is the one published with FlashAttention-4; x must be <= 127.
__device__ __forceinline__ void ex2_poly2(uint64_t x2, float& p0, float& p1) {
    float x0, x1;
    unpack2(x2, x0, x1);
    const uint64_t xc = pack2(fmaxf(x0, -127.0f), fmaxf(x1, -127.0f));
    const uint64_t magic = pack2(12582912.0f, 12582912.0f);  // 2^23 + 2^22
    const uint64_t xr = add2_round_down(xc, magic);           // floor(x) in the low mantissa bits
    const uint64_t xf = sub2(xc, sub2(xr, magic));            // fractional part in [0, 1)
    uint64_t p = fma2(pack2(0.077119089663028717041015625f, 0.077119089663028717041015625f), xf,
                      pack2(0.227564394474029541015625f, 0.227564394474029541015625f));
    p = fma2(p, xf, pack2(0.695146143436431884765625f, 0.695146143436431884765625f));
    p = fma2(p, xf, pack2(1.0f, 1.0f));
    float r0, r1, f0, f1;
    unpack2(xr, r0, r1);
    unpack2(p, f0, f1);
    p0 = __int_as_float((__float_as_int(r0) << 23) + __float_as_int(f0));
    p1 = __int_as_float((__float_as_int(r1) << 23) + __float_as_int(f1));
}

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

}  // namespace ptx
}  // namespace mvoc
