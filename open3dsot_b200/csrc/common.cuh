// open3dsot_b200 — shared device/host helpers for the sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define O3D_OK 0
#define O3D_ERR_ARG (-1)      // bad shape / null pointer / unsupported size
#define O3D_ERR_ALIGN (-2)    // pointer not aligned as the entry point requires
#define O3D_ERR_CUDA (-3)     // a CUDA runtime call failed (see o3d_last_error)

void o3d_set_error(const char* fmt, ...);

#define O3D_REQUIRE(cond, code, ...)                 \
    do {                                             \
        if (!(cond)) {                               \
            o3d_set_error(__VA_ARGS__);              \
            return (code);                           \
        }                                            \
    } while (0)

#define O3D_CHECK_LAUNCH(name)                                                        \
    do {                                                                              \
        cudaError_t e__ = cudaGetLastError();                                         \
        if (e__ != cudaSuccess) {                                                     \
            o3d_set_error("%s: launch failed: %s", name, cudaGetErrorString(e__));    \
            return O3D_ERR_CUDA;                                                      \
        }                                                                             \
    } while (0)

#define O3D_CUDA(call, name)                                                          \
    do {                                                                              \
        cudaError_t e__ = (call);                                                     \
        if (e__ != cudaSuccess) {                                                     \
            o3d_set_error("%s: %s", name, cudaGetErrorString(e__));                   \
            return O3D_ERR_CUDA;                                                      \
        }                                                                             \
    } while (0)

static inline int o3d_num_sms() {
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
    }
    return sms;
}

// upstream cuda_utils.h: opt_n_threads(work) = clamp(2^floor(log2 work), 1, 512)
static inline int o3d_opt_n_threads(int work) {
    if (work < 1) return 1;
    int p = 0;
    while ((1 << (p + 1)) <= work) ++p;
    int t = 1 << p;
    return t > 512 ? 512 : t;
}

#ifdef __CUDACC__
// Squared distance exactly as nvcc contracts upstream's
//   (a-b)*(a-b) + (c-d)*(c-d) + (e-f)*(e-f)   ->  fma(dz,dz, fma(dy,dy, dx*dx))
// written with explicit intrinsics so ptxas cannot re-associate it.
__device__ __forceinline__ float o3d_sq3(float dx, float dy, float dz) {
    return __fmaf_rn(dz, dz, __fmaf_rn(dy, dy, __fmul_rn(dx, dx)));
}
__device__ __forceinline__ float o3d_dist2(float ax, float ay, float az, float bx, float by, float bz) {
    return o3d_sq3(__fsub_rn(ax, bx), __fsub_rn(ay, by), __fsub_rn(az, bz));
}

// ---- mbarrier + 1-D bulk (TMA) copy global -> shared --------------------------------------------
__device__ __forceinline__ uint32_t o3d_smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void o3d_mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(o3d_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void o3d_fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void o3d_fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void o3d_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(o3d_smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void o3d_mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(o3d_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool o3d_mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(o3d_smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug traps (reported as a launch failure) instead of hanging the GPU.
__device__ __forceinline__ void o3d_mbar_wait(uint64_t* bar, uint32_t parity) {
    for (uint32_t spin = 0; spin < (1u << 28); ++spin)
        if (o3d_mbar_try_wait(bar, parity)) return;
    __trap();
}
// bytes must be a multiple of 16; dst/src 16-byte aligned.  SASS: UBLKCP.
__device__ __forceinline__ void o3d_bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            o3d_smem_u32(smem_dst)),
        "l"(gsrc), "r"(bytes), "r"(o3d_smem_u32(bar))
        : "memory");
}
// Ask the bulk-copy engine to pull a contiguous global range into L2 (no SM-side destination).  The activation
// matrices are read in 64..128-byte column slices per k-block; without this every slice re-opens the DRAM page of
// its row (row = 1 KB), with it DRAM streams each tile once, contiguously, and the slices hit L2.
__device__ __forceinline__ void o3d_prefetch_l2(const void* gptr, size_t bytes) {
    const char* p = static_cast<const char*>(gptr);
    const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    const uintptr_t lo = a & ~(uintptr_t)15;
    size_t n = ((a - lo) + bytes + 15) & ~(size_t)15;
    const char* q = reinterpret_cast<const char*>(lo);
    while (n > 0) {
        const uint32_t c = n > (1u << 20) ? (1u << 20) : (uint32_t)n;
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(q), "r"(c) : "memory");
        q += c;
        n -= c;
    }
}
__device__ __forceinline__ uint32_t o3d_lanemask_lt() {
    uint32_t m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

#endif
