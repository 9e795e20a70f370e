// Peer-to-peer halo exchange for the row-strip tiling of one large frame (BASELINE config 5, SURVEY 8(e) row 3):
// the boundary rows of a strip are STORED DIRECTLY into the neighbouring GPU's receive slot over NVLink by an ordinary
// kernel (peer pointers obtained once through CUDA IPC), followed by a release-store of a sequence number into the
// neighbour's flag word; the neighbour's assemble kernel acquires the flag and builds its halo-extended strip.  No NCCL
// call, no staging `.contiguous()` copy, no host synchronisation on the per-iteration path.
//
//   rank r-1:  [ ... own rows ... ]  --bottom `halo` rows-->  recv slot TOP  of rank r
//   rank r+1:  [ ... own rows ... ]  --top    `halo` rows-->  recv slot BOTTOM of rank r
//
// Protocol per exchange number `seq` (all ranks count exchanges in lock-step):
//   send kernel   : copy my boundary rows into the neighbours' slots of parity seq & 1; every block fences system-wide,
//                   the last block to finish writes `seq` into the neighbours' flags (st.release.sys).
//   assemble kernel (same stream, after the send): wait until both of MY flags are >= seq (ld.acquire.sys), then write
//                   ext = [slot TOP | own rows | slot BOTTOM].
// A slot of parity p is rewritten at exchange seq + 2, which a neighbour can only reach after it has received my data of
// exchange seq + 1, i.e. after my assemble kernel of exchange seq has drained the slot (stream order): no write-after-read
// hazard.  The wait is bounded (about 10 s of globaltimer): a lost neighbour sets an error word instead of hanging the GPU.
// The TV prior's exchange (halo_send_tv_kernel) follows the same protocol; its receiver is the TV strip kernel itself
// (sci_tv.cu), which reads the slots in place in its main and fix-up passes - the last reader before the next send.
#include "sci_common.cuh"

namespace {

__device__ __forceinline__ void st_release_sys(unsigned* p, unsigned v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// blockIdx.y = side (0: my top rows -> upper neighbour, 1: my bottom rows -> lower neighbour)
__global__ void __launch_bounds__(256) halo_send_kernel(const float* __restrict__ own, int planes, int rows, int W, int halo,
                                                        float* up_dst, float* down_dst, unsigned* up_flag, unsigned* down_flag,
                                                        unsigned seq, unsigned* done) {
    const int side = blockIdx.y;
    float* dst = side == 0 ? up_dst : down_dst;
    if (dst != nullptr) {
        const int r0 = side == 0 ? 0 : rows - halo;
        const long per_plane = (long)halo * W, n4 = (long)planes * per_plane / 4;
        for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
            const long e = i * 4, pl = e / per_plane, off = e - pl * per_plane;      // W % 4 == 0: a float4 stays inside a row
            const float4 v = *reinterpret_cast<const float4*>(own + (pl * rows + r0) * W + off);
            *reinterpret_cast<float4*>(dst + e) = v;                                 // store into the PEER's memory
        }
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned total = gridDim.x * gridDim.y;
        if (atomicAdd(done, 1u) == total - 1) {
            *done = 0;                                   // ready for the next exchange (stream-ordered)
            __threadfence_system();
            if (up_flag) st_release_sys(up_flag, seq);
            if (down_flag) st_release_sys(down_flag, seq);
        }
    }
}

// The TV prior's halo: f = x + c_b*b of the boundary rows, formed here and stored straight into the neighbours' slots
// (the receiving TV kernel reads the slots in place, there is no assembled strip).  This file is compiled with FMA
// contraction, so the product and the sum are written as separately rounded ops: the same bits as the TV kernel's load.
__global__ void __launch_bounds__(256) halo_send_tv_kernel(const float* __restrict__ x, const float* __restrict__ b, float c_b,
                                                           int planes, int rows, int W, int halo, float* up_dst, float* down_dst,
                                                           unsigned* up_flag, unsigned* down_flag, unsigned seq, unsigned* done) {
    const int side = blockIdx.y;
    float* dst = side == 0 ? up_dst : down_dst;
    if (dst != nullptr) {
        const int r0 = side == 0 ? 0 : rows - halo;
        const long per_plane = (long)halo * W, n2 = (long)planes * per_plane / 2;
        for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += (long)gridDim.x * blockDim.x) {
            const long e = i * 2, pl = e / per_plane, off = e - pl * per_plane;      // W even: a float2 stays inside a row
            const long src = (pl * rows + r0) * W + off;
            float2 v = *reinterpret_cast<const float2*>(x + src);
            if (b) {
                const float2 bb = *reinterpret_cast<const float2*>(b + src);
                v.x = __fadd_rn(v.x, __fmul_rn(c_b, bb.x));
                v.y = __fadd_rn(v.y, __fmul_rn(c_b, bb.y));
            }
            *reinterpret_cast<float2*>(dst + e) = v;                                 // store into the PEER's memory
        }
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned total = gridDim.x * gridDim.y;
        if (atomicAdd(done, 1u) == total - 1) {
            *done = 0;
            __threadfence_system();
            if (up_flag) st_release_sys(up_flag, seq);
            if (down_flag) st_release_sys(down_flag, seq);
        }
    }
}

__global__ void __launch_bounds__(256) halo_assemble_kernel(const float* __restrict__ own, int planes, int rows, int W, int top,
                                                            int bot, const float* __restrict__ recv_top,
                                                            const float* __restrict__ recv_bot, const unsigned* flag_top,
                                                            const unsigned* flag_bot, unsigned seq, float* __restrict__ ext,
                                                            unsigned* err) {
    if (threadIdx.x == 0) {
        const unsigned long long t0 = globaltimer_ns();
        const unsigned* flags[2] = {top ? flag_top : nullptr, bot ? flag_bot : nullptr};
        for (int s = 0; s < 2; ++s) {
            if (!flags[s]) continue;
            while ((int)(ld_acquire_sys(flags[s]) - seq) < 0) {
                if (globaltimer_ns() - t0 > 10000000000ull) { atomicExch(err, 1u + s); break; }
                __nanosleep(200);
            }
        }
    }
    __syncthreads();
    const int er = top + rows + bot;
    const long n4 = (long)planes * er * W / 4;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
        const long e = i * 4, pl = e / ((long)er * W), off = e - pl * (long)er * W;
        const int r = (int)(off / W), c = (int)(off - (long)r * W);
        const float* src;
        if (r < top)             src = recv_top + ((long)pl * top + r) * W + c;
        else if (r < top + rows) src = own + ((long)pl * rows + (r - top)) * W + c;
        else                     src = recv_bot + ((long)pl * bot + (r - top - rows)) * W + c;
        *reinterpret_cast<float4*>(ext + e) = *reinterpret_cast<const float4*>(src);
    }
}

}  // namespace

extern "C" int sci_p2p_alloc(size_t bytes, void** ptr) {
    SCI_REQUIRE(ptr && bytes > 0, "p2p_alloc");
    cudaError_t e = cudaMalloc(ptr, bytes);
    if (e != cudaSuccess) return sci_fail(SCI_ELAUNCH, "p2p_alloc: cudaMalloc", e);
    e = cudaMemset(*ptr, 0, bytes);
    if (e != cudaSuccess) return sci_fail(SCI_ELAUNCH, "p2p_alloc: cudaMemset", e);
    cudaDeviceSynchronize();
    return SCI_OK;
}

extern "C" int sci_p2p_free(void* ptr) {
    if (ptr) cudaFree(ptr);
    return SCI_OK;
}

extern "C" int sci_p2p_get_handle(void* ptr, void* handle64) {
    SCI_REQUIRE(ptr && handle64, "p2p_get_handle");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    cudaError_t e = cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t*>(handle64), ptr);
    if (e != cudaSuccess) return sci_fail(SCI_ELAUNCH, "p2p_get_handle: cudaIpcGetMemHandle", e);
    return SCI_OK;
}

extern "C" int sci_p2p_open_handle(const void* handle64, void** ptr) {
    SCI_REQUIRE(ptr && handle64, "p2p_open_handle");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, sizeof(h));
    cudaError_t e = cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) return sci_fail(SCI_ELAUNCH, "p2p_open_handle: cudaIpcOpenMemHandle", e);
    return SCI_OK;
}

extern "C" int sci_p2p_close_handle(void* ptr) {
    if (ptr) cudaIpcCloseMemHandle(ptr);
    return SCI_OK;
}

extern "C" int sci_halo_send(const float* own, int planes, int rows, int W, int halo, float* up_dst, float* down_dst,
                             unsigned* up_flag, unsigned* down_flag, unsigned seq, unsigned* done_counter, void* stream) {
    SCI_REQUIRE(own && planes > 0 && rows > 0 && W > 0 && W % 4 == 0 && halo > 0 && halo <= rows && done_counter, "halo_send");
    SCI_REQUIRE((up_dst == nullptr) == (up_flag == nullptr) && (down_dst == nullptr) == (down_flag == nullptr), "halo_send: dst / flag pairs");
    const long n4 = (long)planes * halo * W / 4;
    const int gx = (int)max(1L, min((long)SCI_NUM_SMS * 4, (n4 + 255) / 256));
    halo_send_kernel<<<dim3(gx, 2), 256, 0, sci_stream(stream)>>>(own, planes, rows, W, halo, up_dst, down_dst, up_flag, down_flag,
                                                                  seq, done_counter);
    SCI_CHECK_LAUNCH("halo_send");
    return SCI_OK;
}

extern "C" int sci_halo_send_tv(const float* x, const float* b, float c_b, int planes, int rows, int W, int halo, float* up_dst,
                                float* down_dst, unsigned* up_flag, unsigned* down_flag, unsigned seq, unsigned* done_counter,
                                void* stream) {
    SCI_REQUIRE(x && planes > 0 && rows > 0 && W > 0 && W % 2 == 0 && halo > 0 && halo <= rows && done_counter, "halo_send_tv");
    SCI_REQUIRE((up_dst == nullptr) == (up_flag == nullptr) && (down_dst == nullptr) == (down_flag == nullptr),
                "halo_send_tv: dst / flag pairs");
    const long n2 = (long)planes * halo * W / 2;
    const int gx = (int)max(1L, min((long)SCI_NUM_SMS * 4, (n2 + 255) / 256));
    halo_send_tv_kernel<<<dim3(gx, 2), 256, 0, sci_stream(stream)>>>(x, b, c_b, planes, rows, W, halo, up_dst, down_dst,
                                                                     up_flag, down_flag, seq, done_counter);
    SCI_CHECK_LAUNCH("halo_send_tv");
    return SCI_OK;
}

extern "C" int sci_halo_assemble(const float* own, int planes, int rows, int W, int top, int bot, const float* recv_top,
                                 const float* recv_bot, const unsigned* flag_top, const unsigned* flag_bot, unsigned seq,
                                 float* ext, unsigned* err, void* stream) {
    SCI_REQUIRE(own && ext && err && planes > 0 && rows > 0 && W > 0 && W % 4 == 0 && top >= 0 && bot >= 0, "halo_assemble");
    SCI_REQUIRE((top == 0 || (recv_top && flag_top)) && (bot == 0 || (recv_bot && flag_bot)), "halo_assemble: slots");
    const long n4 = (long)planes * (top + rows + bot) * W / 4;
    const int gx = (int)max(1L, min((long)SCI_NUM_SMS * 8, (n4 + 255) / 256));
    halo_assemble_kernel<<<gx, 256, 0, sci_stream(stream)>>>(own, planes, rows, W, top, bot, recv_top, recv_bot, flag_top, flag_bot,
                                                             seq, ext, err);
    SCI_CHECK_LAUNCH("halo_assemble");
    return SCI_OK;
}
