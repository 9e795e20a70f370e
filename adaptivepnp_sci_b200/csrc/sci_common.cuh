// Shared helpers for the sm_100a kernels of the AdaptivePnP_SCI hot path.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#include "sci_b200.h"

#define SCI_NUM_SMS 148   // B200: 2 dies x 74 SMs

extern thread_local char g_sci_last_error[256];

static inline int sci_fail(int code, const char* what, cudaError_t e = cudaSuccess) {
    snprintf(g_sci_last_error, sizeof(g_sci_last_error), "%s%s%s", what, e != cudaSuccess ? ": " : "",
             e != cudaSuccess ? cudaGetErrorString(e) : "");
    return code;
}

#define SCI_REQUIRE(cond, what) \
    do { if (!(cond)) return sci_fail(SCI_EINVAL, "invalid argument: " what); } while (0)

#define SCI_CHECK_LAUNCH(what) \
    do { cudaError_t e__ = cudaGetLastError(); \
         if (e__ != cudaSuccess) return sci_fail(SCI_ELAUNCH, what, e__); } while (0)

static inline cudaStream_t sci_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// Raises `kernel`'s dynamic shared-memory limit to `bytes` the first time it is launched on the current device.  Later
// calls cost a cudaGetDevice and a scan of the few kernels seen so far: no driver call and no lock on the launch path.
// Kernels beyond the table, and devices >= 64, simply set the attribute on every call.
static inline cudaError_t sci_smem_limit(const void* kernel, int bytes) {
    constexpr int SLOTS = 32;
    static std::atomic<const void*> kernels[SLOTS];
    static std::atomic<uint64_t> devices[SLOTS];       // bit d: the attribute is set on device d
    int dev = 0;
    cudaGetDevice(&dev);
    const uint64_t bit = (dev >= 0 && dev < 64) ? 1ull << dev : 0;
    int i = 0;
    for (; i < SLOTS; ++i) {
        const void* k = kernels[i].load(std::memory_order_acquire);
        if (k == nullptr && kernels[i].compare_exchange_strong(k, kernel)) break;
        if (k == kernel) break;
    }
    if (i < SLOTS && (devices[i].load(std::memory_order_acquire) & bit)) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess && i < SLOTS) devices[i].fetch_or(bit, std::memory_order_release);
    return e;
}

static inline int sci_ceil_div(long a, long b) { return (int)((a + b - 1) / b); }

// Streaming (read-once) 128-bit load: bypass L1 allocation, keep L2.
__device__ __forceinline__ float4 ldg_stream4(const float* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}

// Flag word of the peer-to-peer halo exchange (sci_p2p.cu), read with system-scope acquire semantics, and the
// nanosecond clock its bounded waits are measured with.
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Block-wide fp64 sum; result valid in thread 0. `scratch` holds >= 32 doubles.
__device__ __forceinline__ double block_sum(double v, double* scratch) {
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) scratch[wid] = v;
    __syncthreads();
    double r = 0.0;
    if (wid == 0) {
        const int nw = (blockDim.x + 31) >> 5;
        r = lane < nw ? scratch[lane] : 0.0;
        r = warp_sum(r);
    }
    return r;
}
