// Tensor-core 3x3 convolution for sm_100a: implicit GEMM on tcgen05.mma (TF32 operands, fp32
// accumulators in TMEM) fed by TMA, plus the dispatch of the public conv entry points.
//
// Forward / data-gradient kernel (conv_fwd_tc_kernel)
//   GEMM view per output tile:  D[128 pixels][Cout] = sum over 9 taps x Cin/32 chunks of
//        A[128 pixels][32 ch] (activations, K-major)  x  B[Cout][32 ch]^T (packed weights, K-major)
//   * A tile = one TMA box {32 ch, 16 px, 8 rows, 1 image} of the NHWC activation tensor, shifted by the
//     tap offset; out-of-image coordinates are zero-filled by TMA (= the conv's zero padding); stride-2
//     layers use the tensor map's element strides, so no im2col buffer or gather code exists.
//   * B tile = TMA box {32 ch, Cout, 1 tap} of the packed weights.  Both land in 128B-swizzled shared
//     memory, which is exactly the canonical K-major SWIZZLE_128B UMMA operand layout.
//   * warp roles (256 threads, 1 CTA/SM, persistent over tiles): warp 0 = TMA producer, warp 1 = MMA
//     issuer (one elected thread, 4 x tcgen05.mma of K=8 per stage), warp 2 = TMEM allocator,
//     warps 4-7 = epilogue (tcgen05.ld -> scale/shift/ReLU/skip-add/PixelShuffle/TF32 round -> global).
//   * pipelines: smem ring (full/empty mbarriers) between TMA and MMA; two TMEM accumulator stages
//     (tmem_full/tmem_empty) between MMA and epilogue, so the epilogue of tile i overlaps the MMAs of i+1.
// Weight-gradient kernels (conv_wgrad2_tc_kernel, conv_wgrad3_tc_kernel): see the comments above their definitions.
#include <cuda.h>
#include <cuda_fp16.h>
#include <stdlib.h>

#include "sci_common.cuh"

int sci_conv3x3_ref_launch(const sci_conv_desc* d, void* stream);
int sci_wgrad_ref_launch(const sci_wgrad_desc* d, void* stream);
int sci_wgrad_ref_slots(const sci_wgrad_desc* d);

namespace {

constexpr int TILE_W = 16, TILE_H = 8;      // 128 output pixels per tile = UMMA M
constexpr int KCH = 32;                     // fp32 channels per K chunk = 128 bytes = one swizzle row
constexpr int A_BYTES = TILE_W * TILE_H * KCH * 4;   // 16 KB
constexpr int TC_THREADS = 256;
constexpr int MAX_STAGES = 8;

struct FwdParams {
    const float* scale; const float* shift; const float* residual; float* y;
    int N, H, W, Ho, Wo, Cin, Cout, stride, relu, ps, round_tf32, wsplit, emit_lo;
    int tiles_w, tiles_h, num_tiles, k_chunks, stages, acc_stride, tmem_cols;
    int Cstore;       // fp16 storage: channels per pixel of the stored output tensor
    int ks_last;      // see Fwd2Params
    int rb_in, a_bytes;   // bytes per operand row (64: 32 fp16 channels, SWIZZLE_64B; else 128) and per 128-pixel A tile
    int lo_chunk0;        // > 0: first 32-channel chunk of the activations' remainder half (split accumulators, see the MMA issuer)
    int pdl;              // launched with programmatic stream serialization
    int tps;              // filter taps per pipeline stage: 1, or 3 (one filter row) when three (A, B) tile pairs fit a stage -
                          // the profile of the thin stride-2 layers showed both single-thread loops (producer, issuer)
                          // instruction-bound at ~80-120 instructions per 12 KB stage
};

// ---------------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(dst), "l"(tm), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(dst), "l"(tm), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
// one lane of a fully converged warp (the role loops below are warp-uniform; only the issuing instruction is
// predicated, so addresses and descriptors stay in uniform registers instead of per-MMA ELECT/BRA.U loops)
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum) : "memory");
}
// Shared-memory matrix descriptor, version 1 (sm_100).  layout: 2 = SWIZZLE_128B (K-major operands),
// 1 = SWIZZLE_128B_BASE32B (the only layout tcgen05 accepts for MN-major TF32 operands).
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint64_t layout = 2) {
    return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | (1ull << 46) | (layout << 61);
}
// Same instructions issued by ONE elected lane of a converged warp, with the election folded into the predicate of
// the instruction itself: the surrounding code stays straight-line and warp-uniform (descriptor arithmetic in uniform
// registers, no per-instruction divergence handling), which matters because the single issuing thread is the
// critical path for narrow layers (an N=32 TF32 MMA occupies the tensor pipe for only ~67 cycles).
__device__ __forceinline__ void tc_mma_tf32_elect(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\telect.sync _|q, 0xffffffff;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum) : "memory");
}
template <bool HALF>
__device__ __forceinline__ void tc_mma_elect(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
    if (HALF) {
        asm volatile(
            "{\n\t.reg .pred p, q;\n\telect.sync _|q, 0xffffffff;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum) : "memory");
    } else {
        tc_mma_tf32_elect(d_tmem, adesc, bdesc, idesc, accum);
    }
}
// K-major SWIZZLE_128B descriptor split into its 32-bit halves: the low word carries the start address (>> 4) and
// LBO = 16 B, the high word (SBO = 1024 B, version 1, layout SWIZZLE_128B) never changes.  Advancing an operand by whole
// 16-byte units inside the tile is then ONE 32-bit add on the low word.  The base-offset field stays 0: measured on B200,
// the swizzle XOR is taken from the ABSOLUTE shared-memory address bits, so an advanced descriptor reads what TMA wrote.
constexpr uint32_t DESC_HI_K128 = 0x40004040u;
// K-major SWIZZLE_64B (64-byte operand rows = 32 fp16 channels): SBO = 8 rows x 64 B = 512 B, layout type 4
constexpr uint32_t DESC_HI_K64 = 0x80004020u;
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr) { return ((saddr & 0x3FFFFu) >> 4) | 0x10000u; }
template <bool HALF>
__device__ __forceinline__ void mma_lo(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t idesc, uint32_t accum,
                                       uint32_t desc_hi = DESC_HI_K128) {
    if (HALF) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
            "mov.b64 da, {%1, %5};\n\tmov.b64 db, {%2, %5};\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n\t}"
            ::"r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accum), "r"(desc_hi) : "memory");
    } else {
        asm volatile(
            "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
            "mov.b64 da, {%1, %5};\n\tmov.b64 db, {%2, %5};\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %3, p;\n\t}"
            ::"r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accum), "r"(DESC_HI_K128) : "memory");
    }
}
// instruction descriptor: D = f32, A and B K-major in `fmt` (0 = f16, 2 = tf32), N columns, M = 128
__device__ __forceinline__ uint32_t mma_idesc(bool half, int n) {
    const uint32_t fmt = half ? 0u : 2u;
    return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(n >> 3) << 17) | ((128u >> 4) << 24);
}
__device__ __forceinline__ uint32_t pack_half2(float a, float b) {
    uint32_t r;
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));      // low half <- a
    return r;
}
__device__ __forceinline__ float2 unpack_half2(uint32_t h) {
    float2 f;
    asm("{\n\t.reg .b16 lo, hi;\n\tmov.b32 {lo, hi}, %2;\n\tcvt.f32.f16 %0, lo;\n\tcvt.f32.f16 %1, hi;\n\t}" : "=f"(f.x), "=f"(f.y) : "r"(h));
    return f;
}
__device__ __forceinline__ void tc_commit_elect(uint64_t* bar) {
    asm volatile(
        "{\n\t.reg .pred q;\n\telect.sync _|q, 0xffffffff;\n\t"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[32]) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ float rna_tf32(float v) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
    return __uint_as_float(r);
}

// ---------------------------------------------------------------------------------------------------
// forward / data-gradient kernel
// ---------------------------------------------------------------------------------------------------
template <bool HALF>
__global__ void __launch_bounds__(TC_THREADS, 1)
conv_fwd_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const FwdParams p) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[MAX_STAGES], empty_bar[MAX_STAGES], tfull_bar[2], tempty_bar[2];
    __shared__ uint32_t tmem_slot;
    __shared__ float s_scale[256], s_shift[256];

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t b_bytes = (uint32_t)p.Cout * (uint32_t)p.rb_in;
    const uint32_t a_bytes = (uint32_t)p.a_bytes;
    const uint32_t b_tap = b_bytes * (1u + (uint32_t)p.wsplit);                   // wsplit: tf32 hi + remainder weights
    const uint32_t stage_bytes = (uint32_t)p.tps * (a_bytes + b_tap);             // [A tiles of the stage's taps | their B tiles]

    for (int i = threadIdx.x; i < p.Cout; i += TC_THREADS) {
        s_scale[i] = p.scale ? p.scale[i] : 1.f;
        s_shift[i] = p.shift ? p.shift[i] : 0.f;
    }
    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < p.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(&tfull_bar[a], 1); mbar_init(&tempty_bar[a], 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"((uint32_t)p.tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, tmem_slot, 0);
    const int k_steps = (9 / p.tps) * p.k_chunks;
    // programmatic dependent launch inside inference chains (see conv_fwd2_tc_kernel): the next kernel may start its prologue
    // now; this one touches its activations / outputs only after the previous kernel of the stream has completed
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    if (warp == 0) {
        // ===== TMA producer (warp-uniform loop, one elected lane issues) =====
        if (p.pdl) asm volatile("griddepcontrol.wait;" ::: "memory");
        int stage = 0; uint32_t phase = 0;
        for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
            const int tw = tile % p.tiles_w, th = (tile / p.tiles_w) % p.tiles_h, n = tile / (p.tiles_w * p.tiles_h);
            const int iw0 = tw * TILE_W * p.stride - 1, ih0 = th * TILE_H * p.stride - 1;
            const int kstep_el = HALF ? (p.rb_in >> 1) : KCH;
            for (int tap0 = 0; tap0 < 9; tap0 += p.tps) {
                for (int kc = 0; kc < p.k_chunks; ++kc) {
                    mbar_wait(&empty_bar[stage], phase ^ 1u);
                    if (elect_one()) {
                        mbar_arrive_expect_tx(&full_bar[stage], stage_bytes);
                        const uint32_t a_dst = smem_base + (uint32_t)stage * stage_bytes;
                        const uint32_t b_dst = a_dst + (uint32_t)p.tps * a_bytes;
                        for (int t = 0; t < p.tps; ++t) {
                            const int tap = tap0 + t, r = tap / 3, s = tap - 3 * r;
                            tma_load_4d(a_dst + (uint32_t)t * a_bytes, &tmA, &full_bar[stage], kc * kstep_el, iw0 + s, ih0 + r, n);
                            tma_load_3d(b_dst + (uint32_t)t * b_tap, &tmB, &full_bar[stage], kc * kstep_el, 0, tap);
                            if (p.wsplit) tma_load_3d(b_dst + (uint32_t)t * b_tap + b_bytes, &tmB, &full_bar[stage], kc * kstep_el, 0, tap + 9);
                        }
                    }
                    __syncwarp();
                    if (++stage == p.stages) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (warp-uniform loop, election folded into the instruction predicate) =====
        // instruction descriptor: D=f32, A=B=tf32, K-major both, N = Cout, M = 128
        const uint32_t fmt = HALF ? 0u : 2u;
        const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(p.Cout >> 3) << 17) | ((128u >> 4) << 24);
        const uint64_t desc_hi = p.rb_in == 64 ? umma_desc(0, 16, 512, 4) : umma_desc(0, 16, 1024);
        const int ks_full = p.rb_in >> 5;
        int stage = 0; uint32_t phase = 0; int acc = 0; uint32_t acc_phase = 0;
        for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
            mbar_wait(&tempty_bar[acc], acc_phase ^ 1u);
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + (uint32_t)(acc * p.acc_stride);
            // lo_chunk0 > 0 ("3xTF32" layers): the small products - weights' remainder x anything, weights x activations'
            // remainder (channel chunks >= lo_chunk0) - go to a SECOND accumulator next to the main one and are added in the
            // epilogue: the tensor core truncates when it accumulates, and 432 sequential accumulations into one fp32 value left
            // an error floor that the 16 ADMM iterations of the FFDNet loop amplified to 1.2e-3 at 512x512x8
            const uint32_t d_small = p.lo_chunk0 ? d_tmem + (uint32_t)(p.acc_stride >> 1) : d_tmem;
            uint32_t small_started = p.lo_chunk0 ? 0u : 1u;
            int kc = 0;
            for (int ks = 0; ks < k_steps; ++ks) {
                mbar_wait(&full_bar[stage], phase);
                tc_fence_after();
                const uint32_t a0 = smem_base + (uint32_t)stage * stage_bytes, b0 = a0 + (uint32_t)p.tps * a_bytes;
                const int ksn = (kc == p.k_chunks - 1) ? p.ks_last : ks_full;
                const bool lo_x = p.lo_chunk0 && kc >= p.lo_chunk0;
                for (int t = 0; t < p.tps; ++t) {
                    const uint32_t a_addr = a0 + (uint32_t)t * a_bytes, b_addr = b0 + (uint32_t)t * b_tap;
#pragma unroll
                    for (int k = 0; k < KCH / 8; ++k) {
                        if (k < ksn) {
                            const uint32_t accum = lo_x ? (small_started | (uint32_t)(k != 0)) : (uint32_t)((ks | t | k) != 0);
                            tc_mma_elect<HALF>(lo_x ? d_small : d_tmem, desc_hi | (uint64_t)(((a_addr + k * 32) & 0x3FFFFu) >> 4),
                                               desc_hi | (uint64_t)(((b_addr + k * 32) & 0x3FFFFu) >> 4), idesc, accum);
                        }
                    }
                    if (lo_x) small_started = 1u;
                    if (p.wsplit) {
#pragma unroll
                        for (int k = 0; k < KCH / 8; ++k)
                            tc_mma_elect<HALF>(d_small, desc_hi | (uint64_t)(((a_addr + k * 32) & 0x3FFFFu) >> 4),
                                              desc_hi | (uint64_t)(((b_addr + b_bytes + k * 32) & 0x3FFFFu) >> 4), idesc,
                                              p.lo_chunk0 ? (small_started | (uint32_t)(k != 0)) : 1u);
                        small_started = 1u;
                    }
                }
                tc_commit_elect(&empty_bar[stage]);          // frees the smem slot when these MMAs retire
                if (++stage == p.stages) { stage = 0; phase ^= 1u; }
                if (++kc == p.k_chunks) kc = 0;
            }
            tc_commit_elect(&tfull_bar[acc]);                // accumulator complete -> epilogue
            if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
        }
    } else if (warp >= 4) {
        // ===== epilogue: TMEM -> registers -> global =====
        const int q = warp & 3;                            // TMEM lane quarter this warp may access
        const int m = q * 32 + lane, hh = m / TILE_W, ww = m % TILE_W;
        const int Cq = p.Cout >> 2;
        int acc = 0; uint32_t acc_phase = 0;
        if (p.pdl) asm volatile("griddepcontrol.wait;" ::: "memory");      // residual reads / output writes after the previous kernel
        for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
            const int tw = tile % p.tiles_w, th = (tile / p.tiles_w) % p.tiles_h, n = tile / (p.tiles_w * p.tiles_h);
            const int ho = th * TILE_H + hh, wo = tw * TILE_W + ww;
            const bool valid = ho < p.Ho && wo < p.Wo;
            mbar_wait(&tfull_bar[acc], acc_phase);
            tc_fence_after();
            const uint32_t t_row = tmem_base + (uint32_t)(acc * p.acc_stride) + ((uint32_t)(q * 32) << 16);
            for (int c0 = 0; c0 < p.Cout; c0 += 32) {
                float v[32];
                const int nc = min(32, p.Cout - c0);
                if (nc == 32) tmem_ld32(t_row + c0, v); else tmem_ld16(t_row + c0, v);
                if (p.lo_chunk0) {                       // main + small-products accumulator
                    float v2[32];
                    if (nc == 32) tmem_ld32(t_row + (uint32_t)(p.acc_stride >> 1) + c0, v2); else tmem_ld16(t_row + (uint32_t)(p.acc_stride >> 1) + c0, v2);
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] += v2[j];
                }
                if (HALF) {
                    // fp16 storage: 32 columns = 64 bytes of this pixel's row (stride-2 layers: no residual / shuffle / split)
                    if (valid) {
                        __half* yp = reinterpret_cast<__half*>(p.y) + (((long)n * p.Ho + ho) * p.Wo + wo) * p.Cstore + c0;
#pragma unroll
                        for (int j = 0; j < 32; j += 8) {
                            uint32_t h[4];
#pragma unroll
                            for (int e = 0; e < 4; ++e) {
                                float t0 = v[j + 2 * e] * s_scale[c0 + j + 2 * e] + s_shift[c0 + j + 2 * e];
                                float t1 = v[j + 2 * e + 1] * s_scale[c0 + j + 2 * e + 1] + s_shift[c0 + j + 2 * e + 1];
                                if (p.relu) { t0 = fmaxf(t0, 0.f); t1 = fmaxf(t1, 0.f); }
                                h[e] = pack_half2(t0, t1);
                            }
                            if (j < nc) *reinterpret_cast<uint4*>(yp + j) = make_uint4(h[0], h[1], h[2], h[3]);
                        }
                    }
                } else if (valid) {
                    long o;
                    if (p.ps) {
                        const int qq = c0 / Cq, cc = c0 % Cq;
                        o = (((long)n * 2 * p.Ho + 2 * ho + (qq >> 1)) * 2 * p.Wo + 2 * wo + (qq & 1)) * Cq + cc;
                    } else {
                        o = (((long)n * p.Ho + ho) * p.Wo + wo) * (p.Cout << p.emit_lo) + c0;
                    }
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        if (j >= nc) break;
                        float4 r4 = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (p.residual) r4 = *reinterpret_cast<const float4*>(p.residual + o + j);
                        float out[4], lo[4];
                        const float rr[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            float t = v[j + e] * s_scale[c0 + j + e] + s_shift[c0 + j + e];
                            if (p.relu) t = fmaxf(t, 0.f);
                            t += rr[e];
                            const float hi = p.round_tf32 ? rna_tf32(t) : t;
                            lo[e] = rna_tf32(t - hi);
                            out[e] = hi;
                        }
                        *reinterpret_cast<float4*>(p.y + o + j) = make_float4(out[0], out[1], out[2], out[3]);
                        if (p.emit_lo)      // TF32 remainder of the activation, consumed by the next layer's duplicated weights
                            *reinterpret_cast<float4*>(p.y + o + p.Cout + j) = make_float4(lo[0], lo[1], lo[2], lo[3]);
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty_bar[acc]);
            if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
        }
        if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");    // TMA stores (if any) have landed
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols) : "memory");
    }
}


// ---------------------------------------------------------------------------------------------------
// forward / data-gradient kernel, version 2 (stride-1 layers, Cout <= 128): operand reuse
//   Profile of version 1 (profiles/): tensor pipe 19-43 % active, bound by the L2 -> shared-memory fill rate
//   (~42 B/cycle/SM): every activation element was fetched 9x (once per tap) and the weights once per tile.
//   Version 2 cuts the fill traffic:
//   * tile = 128 consecutive pixels of ONE output row.  For filter row r and channel chunk kc a single TMA box
//     {32 ch, 130 px, 1 row} is loaded; the three horizontal taps s = 0,1,2 are the SAME shared-memory tile read
//     through UMMA descriptors whose start address is advanced by s pixels (s * 128 B; the hardware derives the
//     swizzle phase from the absolute shared-memory address, so shifted views need no re-layout).  Activation fill traffic: 3x per element instead of 9x
//     (the 3 vertical neighbours come from L2).
//   * when all 9 x Cin x Cout weights fit beside the pipeline (<= ~150 KB: every 32/64/96-channel layer of
//     FastDVDnet) they are loaded ONCE per CTA and stay resident; otherwise the three B tiles of a stage are
//     streamed with the row box.
// ---------------------------------------------------------------------------------------------------
constexpr int ROW_PX = 130;
constexpr int ROW_BYTES = ROW_PX * KCH * 4;       // 16640
constexpr int A2_STAGE = 17 * 1024;               // row box rounded up to the 1024-byte swizzle period

struct Fwd2Params {
    const float* scale; const float* shift; const float* residual; float* y;
    int N, H, W, Cin, Cout, relu, ps, round_tf32;
    int tiles_w, num_tiles, k_chunks, stages, acc_stride, tmem_cols, resident, out_bufs;
    const float* planar_in1; float* planar_out;   // fused network output: out[n][c][h][w] = in1[n][c][h][w] - conv[c], c < 3 (MODE 3: 1)
    int pdl;          // launched with programmatic stream serialization: see griddepcontrol below
    int col0, Ctot;   // this launch computes GEMM columns [col0, col0 + Cout) of a layer with Ctot columns (Cout = 256 layers run as two halves)
    int stack;        // filter rows stacked along N (see the MMA issuer); needs resident weights, R >= 2, 3*Cout <= 256
    int R, tiles_h;   // rows per super-tile (R output rows share their R+2 input rows), super-tiles per image column strip
    int dbg;   // SCI_CONV_DBG timing experiments (results invalid): 1 = no MMAs, 2 = no activation loads, 4 = no stores
    // fp16 storage (HALF kernels): a 128-byte operand row holds 64 channels.  One epilogue unit = `ucols` accumulator columns
    // (64, or 32 when the layer / its PixelShuffle sub-pixel group has 32 real channels) -> ONE 64-channel fp16 pixel row of
    // the stored tensor (the missing half is written as zeros); Cstore = channels per pixel of the stored output tensor
    int ucols, Cstore;
    // MODE 4 (data gradient + activation backward of the layer that PRODUCED this tensor, fused): dz = (conv [+ residual]) *
    // (mask_y > 0); col_s1[c] += sum dz, col_s2[c] += sum dz * mask_y  (bias / BatchNorm gradients), see the epilogue.
    // MODE 5 = MODE 4 with fixed-order sums: col_s1 is then slot 0 of this launch's [grid][2][ncol] workspace slots (ncol =
    // stored channels) and col_s2 only says whether the second sums are wanted
    const float* mask_y; float* col_s1; float* col_s2; int mask_relu;
    // split > 0 (HALF, FFDNet inference at ~fp32 accuracy): every activation and weight travels as fp16 value + fp16 remainder
    // scaled by 2^11; a 64-channel chunk is [32 values | their 32 remainders].  Per chunk the issuer multiplies value x value
    // into the main accumulator and value x remainder + remainder x value into a second one (columns + Cout), the epilogue
    // adds them (x 2^-11), applies the layer's epilogue and emits the same split form.  split = value K steps per chunk (1, 2).
    int split;
    int ks_last;      // K steps (8 fp32 / 16 fp16 channels each) of the LAST channel chunk that can hold non-zero channels (1..4):
                      // zero-padded K columns are not multiplied (12 -> 90: 28 of 64 fp16 channels used -> 2 of 4 steps)
    // fp16 tensors with 32 channels are stored as 64-byte pixel rows (no zero half): operand rows / staging rows of 64 bytes use the
    // SWIZZLE_64B layouts.  rb_in / rb_out = bytes per pixel row of the input operand / of the stored output (64 or 128)
    int rb_in, rb_out, a_stage, row_bytes;
    uint32_t desc_hi;
};

// Epilogue organisation (round 2).  The ncu source view of the full-resolution layers showed the four epilogue warps
// - one per SM sub-partition - busy >90 % of the time at IPC 0.25 (407 instructions per 32-channel chunk, every one
// waiting for its predecessor) while the MMA warp sat on the tmem_empty barrier: the 12->90 layer was bound by its
// epilogue, not by the tensor pipe, shared memory or HBM.  Hence
//   * EPI_WG = 2 epilogue warpgroups (warps 4-7 and 8-11; a warp may only touch the TMEM lane quarter warp % 4, so the
//     second group shares the quarters and takes every second (row, chunk) unit): two warps per scheduler hide each
//     other's latencies;
//   * MODE selects the epilogue at compile time (0 = TMA store, 1 = TMA store + skip-add, 2 = fused planar network
//     output of 3 planes, 3 = the same with 1 plane (gray), 4 = data gradient with the fused activation backward, 5 = the
//     same with fixed-order column sums) instead of run-time flags per element; scale / shift come from shared memory as float4;
//   * the planar mode fetches the in1 values of ALL its rows before it waits for the accumulator (the per-row prefetch
//     left the HBM latency of those loads exposed: 46 % of the epilogue's samples in the 32->3 layer).
//   * HALF: fp16 storage and operands (kind::f16, fp32 accumulation): the same 11-bit significand as TF32 - the products
//     are as exact - at half the bytes per channel and twice the tensor rate.  Used for inference chains; the training
//     passes keep fp32 activations (the weight-gradient kernels read them).
template <int EPI_WG, int MODE, bool HALF>
__global__ void __launch_bounds__(128 + 128 * EPI_WG, 1)
conv_fwd2_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                    const __grid_constant__ CUtensorMap tmY, const Fwd2Params p) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[MAX_STAGES], empty_bar[MAX_STAGES], tfull_bar[2], tempty_bar[2], w_bar;
    __shared__ uint32_t tmem_slot;
    __shared__ __align__(16) float s_scale[128], s_shift[128];
    __shared__ float s_cs1[MODE == 4 ? 128 : 1], s_cs2[MODE == 4 ? 128 : 1];      // CTA partial column sums (MODE 4)
    __shared__ float s_wcs[MODE == 5 ? 4 * EPI_WG : 1][2][128];                    // per epilogue warp (MODE 5)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (MODE == 4) {
        for (int i = threadIdx.x; i < 128; i += 128 + 128 * EPI_WG) { s_cs1[i] = 0.f; s_cs2[i] = 0.f; }
    }
    if (MODE == 5) {
        for (int i = threadIdx.x; i < 4 * EPI_WG * 2 * 128; i += 128 + 128 * EPI_WG) (&s_wcs[0][0][0])[i] = 0.f;
    }
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t b_bytes = (uint32_t)p.Cout * (uint32_t)p.rb_in;
    const uint32_t w_bytes = p.resident ? 9u * (uint32_t)p.k_chunks * b_bytes : 0u;
    // streamed weights with two output rows per tile (wpair): a stage carries BOTH input rows a filter row needs
    const bool wpair = !p.resident && p.R == 2;
    const uint32_t stage_bytes = (uint32_t)p.a_stage * (wpair ? 2u : 1u) + (p.resident ? 0u : 3u * b_bytes);
    const uint32_t ring_base = smem_base + w_bytes;
    const uint32_t stage_out_base = ring_base + (uint32_t)p.stages * stage_bytes;   // 4 EPI_WG warps x out_bufs x 4 KB store staging

    for (int i = threadIdx.x; i < p.Cout; i += 128 + 128 * EPI_WG) {
        s_scale[i] = p.scale ? p.scale[p.col0 + i] : 1.f;
        s_shift[i] = p.shift ? p.shift[p.col0 + i] : 0.f;
    }
    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < p.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(&tfull_bar[a], 1); mbar_init(&tempty_bar[a], 4 * EPI_WG); }
        mbar_init(&w_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"((uint32_t)p.tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, tmem_slot, 0);
    // the next kernel of the stream may be scheduled as soon as SMs free up (it waits for our completion itself)
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    if (warp == 0) {
        // ===== TMA producer (warp-uniform loop, one elected lane issues) =====
        if (p.resident) {
            if (elect_one()) {
                mbar_arrive_expect_tx(&w_bar, w_bytes);
                for (int tap = 0; tap < 9; ++tap)
                    for (int kc = 0; kc < p.k_chunks; ++kc) {
                        // default: tiles ordered [tap][kc]; stacked: [s][kc][r] so that the three filter rows of a
                        // horizontal tap form ONE K-major B matrix of 3*Cout rows
                        const uint32_t slot = p.stack ? (uint32_t)(((tap % 3) * p.k_chunks + kc) * 3 + tap / 3)
                                                      : (uint32_t)(tap * p.k_chunks + kc);
                        tma_load_3d(smem_base + slot * b_bytes, &tmB, &w_bar, kc * (HALF ? (p.rb_in >> 1) : KCH), p.col0, tap);
                    }
            }
            __syncwarp();
        }
        // Programmatic dependent launch: everything above (barriers, TMEM, tensor maps, the resident WEIGHTS, which no
        // kernel of the running chain writes) overlapped the tail of the previous kernel; its activations may only be
        // read once it has completed and flushed
        if (p.pdl) asm volatile("griddepcontrol.wait;" ::: "memory");
        int stage = 0; uint32_t phase = 0;
        for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
            const int wt = tile % p.tiles_w, hg = (tile / p.tiles_w) % p.tiles_h, n = tile / (p.tiles_w * p.tiles_h);
            const int y0 = hg * p.R, rows = min(p.R, p.H - y0);
            if (wpair) {
                // Streamed weights, two output rows per tile: per (filter row r, channel chunk) ONE stage holds the weight tiles of
                // the three horizontal taps and the two input rows y0 + r - 1, y0 + r they multiply - the weight fill per output
                // row halves (the 128-channel layers were bound by it: 390 KB per row tile at ~42 B/cycle/SM from L2)
                for (int r = 0; r < 3; ++r) {
                    for (int kc = 0; kc < p.k_chunks; ++kc) {
                        mbar_wait(&empty_bar[stage], phase ^ 1u);
                        if (elect_one()) {
                            mbar_arrive_expect_tx(&full_bar[stage], 2u * (uint32_t)p.row_bytes + 3u * b_bytes);
                            const uint32_t a_dst = ring_base + (uint32_t)stage * stage_bytes;
                            const int cc = kc * (HALF ? (p.rb_in >> 1) : KCH);
                            tma_load_4d(a_dst, &tmA, &full_bar[stage], cc, wt * 128 - 1, y0 + r - 1, n);
                            tma_load_4d(a_dst + (uint32_t)p.a_stage, &tmA, &full_bar[stage], cc, wt * 128 - 1, y0 + r, n);
                            for (int s = 0; s < 3; ++s)
                                tma_load_3d(a_dst + 2u * (uint32_t)p.a_stage + (uint32_t)s * b_bytes, &tmB, &full_bar[stage], cc, p.col0, r * 3 + s);
                        }
                        __syncwarp();
                        if (++stage == p.stages) { stage = 0; phase ^= 1u; }
                    }
                }
                continue;
            }
            // input rows y0-1 .. y0+rows: row j feeds output row t = j - r as filter row r (R = 1: j is the filter row)
            for (int j = 0; j < rows + 2; ++j) {
                for (int kc = 0; kc < p.k_chunks; ++kc) {
                    mbar_wait(&empty_bar[stage], phase ^ 1u);
                    if (elect_one()) {
                        const bool skip_a = (p.dbg & 2) != 0;
                        mbar_arrive_expect_tx(&full_bar[stage], (skip_a ? 0u : (uint32_t)p.row_bytes) + (p.resident ? 0u : 3u * b_bytes));
                        const uint32_t a_dst = ring_base + (uint32_t)stage * stage_bytes;
                        if (!skip_a) tma_load_4d(a_dst, &tmA, &full_bar[stage], kc * (HALF ? (p.rb_in >> 1) : KCH), wt * 128 - 1, y0 + j - 1, n);
                        if (!p.resident) {       // streamed weights: R == 1, j is the filter row
                            for (int s = 0; s < 3; ++s)
                                tma_load_3d(a_dst + (uint32_t)p.a_stage + (uint32_t)s * b_bytes, &tmB, &full_bar[stage], kc * (HALF ? (p.rb_in >> 1) : KCH), p.col0, j * 3 + s);
                        }
                    }
                    __syncwarp();
                    if (++stage == p.stages) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        // Round 2: the ncu source view showed this warp as the critical path of EVERY layer: ~15 SASS instructions per
        // UTCHMMA (ELECT + VOTEU per instruction, 64-bit descriptor arithmetic in vector registers, four R2UR) at ~6 cycles
        // each = ~100 cycles per MMA, against 40-64 cycles of shared-memory operand reads (N = 32..128).  Now: all lanes wait
        // on the barriers (warp-uniform), ONE lane elected once issues a stage's MMAs in straight-line code; descriptors are
        // a per-stage 32-bit low word plus compile-time increments, the high word is a constant.
        const bool leader = elect_one();
        const uint32_t idesc = mma_idesc(HALF, p.Cout);
        if (p.resident) { mbar_wait(&w_bar, 0); tc_fence_after(); }
        int stage = 0; uint32_t phase = 0; int acc = 0; uint32_t acc_phase = 0;
        const uint32_t b_tile_lo = b_bytes >> 4;                  // one [Cout][32 ch] weight tile, in descriptor units
        const uint32_t tapu = (uint32_t)p.rb_in >> 4;             // one pixel (= one horizontal tap) in 16-byte descriptor units
        const int ks_full = p.rb_in >> 5;                         // 32-byte K steps per operand row
        for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
            mbar_wait(&tempty_bar[acc], acc_phase ^ 1u);
            tc_fence_after();
            const int hg = (tile / p.tiles_w) % p.tiles_h;
            const int rows = min(p.R, p.H - hg * p.R);
            const uint32_t d_base = tmem_base + (uint32_t)(acc * p.R * p.acc_stride);
            if (p.R == 1) {
                // one output row per tile (streamed or resident weights)
                for (int r = 0; r < 3; ++r) {
                    for (int kc = 0; kc < p.k_chunks; ++kc) {
                        mbar_wait(&full_bar[stage], phase);
                        tc_fence_after();
                        if (leader) {
                            const uint32_t a_addr = ring_base + (uint32_t)stage * stage_bytes;
                            const uint32_t a_lo = desc_lo(a_addr);
                            const int ksn = (kc == p.k_chunks - 1) ? p.ks_last : ks_full;     // K steps that can hold non-zero channels
                            const uint32_t b_lo = desc_lo(p.resident ? smem_base + (uint32_t)(r * 3 * p.k_chunks + kc) * b_bytes : a_addr + (uint32_t)p.a_stage);
                            const uint32_t b_step = p.resident ? (uint32_t)p.k_chunks * b_tile_lo : b_tile_lo;
                            const uint32_t first = (uint32_t)((r | kc) != 0);
                            if (HALF && p.split) {
                                // chunk = [values (K steps 0,1) | remainders * 2^11 (K steps 2,3)] on both operands
                                const uint32_t d_small = d_base + (uint32_t)p.Cout;
#pragma unroll
                                for (int s = 0; s < 3; ++s) {
#pragma unroll
                                    for (int k = 0; k < 2; ++k) {
                                        if (k < p.split) {
                                            const uint32_t a_v = a_lo + s * tapu + k * 2, b_v = b_lo + s * b_step + k * 2;
                                            mma_lo<HALF>(d_base, a_v, b_v, idesc, (s | k) ? 1u : first, p.desc_hi);          // value x value
                                            mma_lo<HALF>(d_small, a_v, b_v + 4, idesc, (s | k) ? 1u : first, p.desc_hi);     // value x weight remainder
                                            mma_lo<HALF>(d_small, a_v + 4, b_v, idesc, 1u, p.desc_hi);                       // remainder x weight value
                                        }
                                    }
                                }
                            } else if (!(p.dbg & 1)) {
#pragma unroll
                                for (int s = 0; s < 3; ++s) {
#pragma unroll
                                    for (int k = 0; k < KCH / 8; ++k)
                                        if (k < ksn) mma_lo<HALF>(d_base, a_lo + s * tapu + k * 2, b_lo + s * b_step + k * 2, idesc, (s | k) ? 1u : first, p.desc_hi);
                                }
                            }
                            tc_commit(&empty_bar[stage]);
                        }
                        __syncwarp();
                        if (++stage == p.stages) { stage = 0; phase ^= 1u; }
                    }
                }
            } else if (wpair) {
                for (int r = 0; r < 3; ++r) {
                    for (int kc = 0; kc < p.k_chunks; ++kc) {
                        mbar_wait(&full_bar[stage], phase);
                        tc_fence_after();
                        if (leader) {
                            const uint32_t a_addr = ring_base + (uint32_t)stage * stage_bytes;
                            const int ksn = (kc == p.k_chunks - 1) ? p.ks_last : ks_full;
                            const uint32_t b_lo = desc_lo(a_addr + 2u * (uint32_t)p.a_stage);
                            const uint32_t first = (uint32_t)((r | kc) != 0);
                            if (!(p.dbg & 1)) {
                                for (int t = 0; t < rows; ++t) {        // input row y0 + r - 1 + t is filter row r of output row t
                                    const uint32_t a_lo = desc_lo(a_addr + (uint32_t)t * (uint32_t)p.a_stage);
                                    const uint32_t d_tmem = d_base + (uint32_t)(t * p.acc_stride);
#pragma unroll
                                    for (int s = 0; s < 3; ++s) {
#pragma unroll
                                        for (int k = 0; k < KCH / 8; ++k)
                                            if (k < ksn) mma_lo<HALF>(d_tmem, a_lo + s * tapu + k * 2, b_lo + s * b_tile_lo + k * 2, idesc, (s | k) ? 1u : first, p.desc_hi);
                                    }
                                }
                            }
                            tc_commit(&empty_bar[stage]);
                        }
                        __syncwarp();
                        if (++stage == p.stages) { stage = 0; phase ^= 1u; }
                    }
                }
            } else if (p.stack) {
                // Filter rows stacked along N.  Input row j (relative to y0 - 1) is filter row r of output row t = j - r; the
                // accumulators of the super-tile sit in REVERSE row order (row t at column (R-1-t)*Cout), so ONE MMA with
                // B = [W(r_lo) | .. | W(r_hi)] (N = nr*Cout) adds the row's contribution to all output rows it touches.
                // The A operand (128 px x 8 ch, the shared-memory-bandwidth cost of a TF32 MMA) is then read once per
                // horizontal tap instead of once per (tap, filter row): ~1.5-1.8x fewer tensor-pipe cycles for Cout = 32/64.
                for (int j = 0; j < rows + 2; ++j) {
                    const int r_lo = max(0, j - (rows - 1)), r_hi = min(2, j);
                    const int nr = r_hi - r_lo + 1;
                    const uint32_t d_col = d_base + (uint32_t)((p.R - 1 - (j - r_lo)) * p.acc_stride);
                    const uint32_t idesc_n = (idesc & ~(0x3Fu << 17)) | ((uint32_t)((nr * p.Cout) >> 3) << 17);
                    const uint32_t idesc_m = (idesc & ~(0x3Fu << 17)) | ((uint32_t)(((nr - 1) * p.Cout) >> 3) << 17);
                    for (int kc = 0; kc < p.k_chunks; ++kc) {
                        mbar_wait(&full_bar[stage], phase);
                        tc_fence_after();
                        if (leader) {
                            const uint32_t a_lo = desc_lo(ring_base + (uint32_t)stage * stage_bytes);
                            const int ksn = (kc == p.k_chunks - 1) ? p.ks_last : ks_full;
                            // weight tiles ordered [s][kc][r]: the three filter rows of tap s are consecutive
                            const uint32_t b_lo = desc_lo(smem_base + (uint32_t)(kc * 3 + r_lo) * b_bytes);
                            const uint32_t b_step = (uint32_t)(3 * p.k_chunks) * b_tile_lo;
                            if (p.dbg & 1) {
                            } else if (r_lo == 0 && kc == 0) {
                                // this row opens the accumulator of output row t = j (r = 0): that slice must overwrite
                                mma_lo<HALF>(d_col, a_lo, b_lo, idesc, 0u, p.desc_hi);
                                if (nr > 1) mma_lo<HALF>(d_col + (uint32_t)p.acc_stride, a_lo, b_lo + b_tile_lo, idesc_m, 1u, p.desc_hi);
#pragma unroll
                                for (int sk = 1; sk < 3 * (KCH / 8); ++sk) {
                                    const int s = sk / (KCH / 8), k = sk % (KCH / 8);
                                    if (k < ksn) mma_lo<HALF>(d_col, a_lo + s * tapu + k * 2, b_lo + s * b_step + k * 2, idesc_n, 1u, p.desc_hi);
                                }
                            } else {
#pragma unroll
                                for (int s = 0; s < 3; ++s) {
#pragma unroll
                                    for (int k = 0; k < KCH / 8; ++k)
                                        if (k < ksn) mma_lo<HALF>(d_col, a_lo + s * tapu + k * 2, b_lo + s * b_step + k * 2, idesc_n, 1u, p.desc_hi);
                                }
                            }
                            tc_commit(&empty_bar[stage]);
                        }
                        __syncwarp();
                        if (++stage == p.stages) { stage = 0; phase ^= 1u; }
                    }
                }
            } else {
                for (int j = 0; j < rows + 2; ++j) {
                    for (int kc = 0; kc < p.k_chunks; ++kc) {
                        mbar_wait(&full_bar[stage], phase);
                        tc_fence_after();
                        if (leader) {
                            const uint32_t a_addr = ring_base + (uint32_t)stage * stage_bytes;
                            const uint32_t a_lo = desc_lo(a_addr);
                            const int ksn = (kc == p.k_chunks - 1) ? p.ks_last : ks_full;
                            // the loaded input row is filter row r = j - t of every output row t of the super-tile it touches
                            for (int t = max(0, j - 2); t <= min(rows - 1, j); ++t) {
                                const int r = j - t;
                                const uint32_t d_tmem = d_base + (uint32_t)(t * p.acc_stride);
                                const uint32_t b_lo = desc_lo(p.resident ? smem_base + (uint32_t)(r * 3 * p.k_chunks + kc) * b_bytes : a_addr + (uint32_t)p.a_stage);
                                const uint32_t b_step = p.resident ? (uint32_t)p.k_chunks * b_tile_lo : b_tile_lo;
                                const uint32_t first = (uint32_t)((r | kc) != 0);
                                if (!(p.dbg & 1)) {
#pragma unroll
                                    for (int s = 0; s < 3; ++s) {
#pragma unroll
                                        for (int k = 0; k < KCH / 8; ++k)
                                            if (k < ksn) mma_lo<HALF>(d_tmem, a_lo + s * tapu + k * 2, b_lo + s * b_step + k * 2, idesc, (s | k) ? 1u : first, p.desc_hi);
                                    }
                                }
                            }
                            tc_commit(&empty_bar[stage]);
                        }
                        __syncwarp();
                        if (++stage == p.stages) { stage = 0; phase ^= 1u; }
                    }
                }
            }
            if (leader) tc_commit(&tfull_bar[acc]);
            __syncwarp();
            if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
        }
    } else if (warp >= 4) {
        // ===== epilogue: TMEM -> registers -> (scale/shift, ReLU, skip-add, TF32 round) -> swizzled staging -> TMA store
        const int q = warp & 3;                            // TMEM lane quarter this warp may access
        const int g = (warp >> 2) - 1;                     // epilogue warpgroup: takes the units u = g (mod EPI_WG)
        const int m = q * 32 + lane;
        const int Cq = p.Ctot >> 2;
        const int nch = p.Cout >> 5;                       // 32-column chunks per output row
        const float lower = p.relu ? 0.f : -INFINITY;
        const long pl_plane = (long)p.H * p.W;
        constexpr bool PLANAR = MODE == 2 || MODE == 3;
        constexpr int NPL = MODE == 3 ? 1 : 3;                // planes per frame of the planar output
        constexpr int PIN_ROWS = (8 + EPI_WG - 1) / EPI_WG;   // planar mode: rows of a super-tile (R <= 8) per warpgroup
        const uint32_t tile_b = (uint32_t)p.rb_out * 32u;      // staging tile of a warp: 32 pixel rows of the stored output
        const uint32_t sbuf0 = stage_out_base + (uint32_t)((g * 4 + q) * p.out_bufs) * tile_b;
        int acc = 0; uint32_t acc_phase = 0;
        uint32_t st_cnt = 0;
        if (p.pdl) asm volatile("griddepcontrol.wait;" ::: "memory");      // residual / in1 come from earlier kernels
        for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
            const int wt = tile % p.tiles_w, hg = (tile / p.tiles_w) % p.tiles_h, n = tile / (p.tiles_w * p.tiles_h);
            const int y0 = hg * p.R, rows = min(p.R, p.H - y0);
            const int wo = wt * 128 + m;
            const bool valid = wo < p.W;
            const int units = rows * nch;
            // element offset of this lane's 32-channel segment of chunk c0 of output row ho in the output / residual tensor
            auto out_offset = [&](int ho, int c0) -> long {
                const int cg = p.col0 + c0;                           // column of the whole layer
                if (p.ps) {
                    const int qq = cg / Cq, cc = cg % Cq;
                    return (((long)n * 2 * p.H + 2 * ho + (qq >> 1)) * 2 * p.W + 2 * wo + (qq & 1)) * Cq + cc;
                }
                return (((long)n * p.H + ho) * p.W + wo) * p.Ctot + cg;
            };
            // operands from global memory are requested while the MMAs of this tile are still running
            float4 rr[8];
            float pin[PIN_ROWS][3];
            if (!HALF && MODE == 1) {
#pragma unroll
                for (int j = 0; j < 8; ++j) rr[j] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (p.residual && valid && g < units) {
                    const float4* rp = reinterpret_cast<const float4*>(p.residual + out_offset(y0 + g / nch, (g % nch) << 5));
#pragma unroll
                    for (int j = 0; j < 8; ++j) rr[j] = __ldg(rp + j);
                }
            }
            if (PLANAR) {
#pragma unroll
                for (int i = 0; i < PIN_ROWS; ++i) {
                    const int t = g + i * EPI_WG;
#pragma unroll
                    for (int c = 0; c < 3; ++c) pin[i][c] = 0.f;
                    if (valid && t < rows) {
                        const long o = (long)n * NPL * pl_plane + (long)(y0 + t) * p.W + wo;
#pragma unroll
                        for (int c = 0; c < NPL; ++c) pin[i][c] = __ldg(p.planar_in1 + o + c * pl_plane);
                    }
                }
            }
            mbar_wait(&tfull_bar[acc], acc_phase);
            tc_fence_after();
            if (HALF && !PLANAR) {
                // ---- fp16 output: unit = `ucols` accumulator columns -> one 64-channel (128-byte) pixel row
                const int nun = (p.Cout + p.ucols - 1) / p.ucols;
                const int hunits = rows * nun;
                // skip values of unit u (fp16, up to 128 bytes of this lane's pixel row), requested one unit ahead
                auto load_res = [&](int u, uint4 (&r)[8]) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) r[j] = make_uint4(0u, 0u, 0u, 0u);
                    if (u < hunits && valid) {
                        const int t = u / nun, col0 = (u - t * nun) * p.ucols;
                        const int ncv = min(p.ucols, p.Cout - col0);
                        const int cg = p.col0 + col0, ho = y0 + t;
                        int qq = 0, cx = cg;
                        if (p.ps) { qq = cg / Cq; cx = cg - qq * Cq; }
                        const long pix = p.ps ? (((long)n * 2 * p.H + 2 * ho + (qq >> 1)) * 2 * p.W + 2 * wo + (qq & 1))
                                              : (((long)n * p.H + ho) * p.W + wo);
                        const uint4* rp = reinterpret_cast<const uint4*>(reinterpret_cast<const __half*>(p.residual) + pix * p.Cstore + cx);
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            if (j * 8 < ncv) r[j] = __ldg(rp + j);
                    }
                };
                uint4 rres[8];
                if (MODE == 1) load_res(g, rres);
                for (int u = g; u < hunits; u += EPI_WG) {
                    const int t = u / nun, col0 = (u - t * nun) * p.ucols;
                    const int ncv = min(p.ucols, p.Cout - col0);           // valid accumulator columns of this unit (32 or 64)
                    const int ho = y0 + t;
                    const int cg = p.col0 + col0;
                    int qq = 0, cx = cg;
                    if (p.ps) { qq = cg / Cq; cx = cg - qq * Cq; }
                    uint4 rnext[8];
                    if (MODE == 1) load_res(u + EPI_WG, rnext);
                    const uint32_t t_row = tmem_base + (uint32_t)((acc * p.R + (p.stack ? p.R - 1 - t : t)) * p.acc_stride) + ((uint32_t)(q * 32) << 16);
                    uint32_t hv[32];                                        // 64 fp16 values of this lane's pixel
                    if (p.split) {
                        // main + 2^-11 * small -> epilogue -> [32 fp16 values | 32 remainders * 2^11] = one 64-channel stored chunk
                        float v[32], sm[32];
                        tmem_ld32(t_row + col0, v);
                        tmem_ld32(t_row + p.Cout + col0, sm);
#pragma unroll
                        for (int j = 0; j < 32; j += 2) {
                            const float a0 = fmaxf(fmaf(fmaf(sm[j], 1.f / 2048.f, v[j]), s_scale[col0 + j], s_shift[col0 + j]), lower);
                            const float a1 = fmaxf(fmaf(fmaf(sm[j + 1], 1.f / 2048.f, v[j + 1]), s_scale[col0 + j + 1], s_shift[col0 + j + 1]), lower);
                            const uint32_t h = pack_half2(a0, a1);
                            const float2 hf = unpack_half2(h);
                            hv[j >> 1] = h;
                            hv[16 + (j >> 1)] = pack_half2((a0 - hf.x) * 2048.f, (a1 - hf.y) * 2048.f);
                        }
                        cx = 2 * cg;                                        // stored chunk of this 32-column group
                    } else
#pragma unroll
                    for (int hb = 0; hb < 2; ++hb) {
                        if (hb * 32 < ncv) {
                            float v[32];
                            tmem_ld32(t_row + col0 + hb * 32, v);
#pragma unroll
                            for (int j = 0; j < 32; j += 4) {
                                const float4 sc = *reinterpret_cast<const float4*>(&s_scale[col0 + hb * 32 + j]);
                                const float4 sh = *reinterpret_cast<const float4*>(&s_shift[col0 + hb * 32 + j]);
                                float a0 = fmaxf(fmaf(v[j], sc.x, sh.x), lower), a1 = fmaxf(fmaf(v[j + 1], sc.y, sh.y), lower);
                                float a2 = fmaxf(fmaf(v[j + 2], sc.z, sh.z), lower), a3 = fmaxf(fmaf(v[j + 3], sc.w, sh.w), lower);
                                if (MODE == 1) {
                                    const uint4 r4 = rres[hb * 4 + (j >> 3)];
                                    const float2 r0 = unpack_half2((j & 4) ? r4.z : r4.x), r1 = unpack_half2((j & 4) ? r4.w : r4.y);
                                    a0 += r0.x; a1 += r0.y; a2 += r1.x; a3 += r1.y;
                                }
                                hv[hb * 16 + (j >> 1)] = pack_half2(a0, a1);
                                hv[hb * 16 + (j >> 1) + 1] = pack_half2(a2, a3);
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < 16; ++j) hv[hb * 16 + j] = 0u;
                        }
                    }
                    const uint32_t sbuf = sbuf0 + (p.out_bufs == 2 ? (st_cnt & 1) * tile_b : 0u);
                    if (lane == 0) {
                        if (p.out_bufs == 2) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
                        else                 asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                    }
                    __syncwarp();
                    if (p.rb_out == 64) {
                        // 32-channel tensor: 64-byte pixel rows, SWIZZLE_64B (16-byte chunk j of row l at j ^ ((l >> 1) & 3))
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const uint32_t a = sbuf + (uint32_t)lane * 64u + (uint32_t)((j ^ ((lane >> 1) & 3)) << 4);
                            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(hv[4 * j]), "r"(hv[4 * j + 1]), "r"(hv[4 * j + 2]), "r"(hv[4 * j + 3]) : "memory");
                        }
                    } else {
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const uint32_t a = sbuf + (uint32_t)lane * 128u + (uint32_t)((j ^ (lane & 7)) << 4);
                            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(hv[4 * j]), "r"(hv[4 * j + 1]), "r"(hv[4 * j + 2]), "r"(hv[4 * j + 3]) : "memory");
                        }
                    }
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) {
                        int cw = wt * 128 + q * 32, chh = ho;
                        if (p.ps) { cw = 2 * cw + (qq & 1); chh = 2 * ho + (qq >> 1); }
                        asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                                     ::"l"(&tmY), "r"(sbuf), "r"(cx), "r"(cw), "r"(chh), "r"(n) : "memory");
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    }
                    ++st_cnt;
                    if (MODE == 1) {
#pragma unroll
                        for (int j = 0; j < 8; ++j) rres[j] = rnext[j];
                    }
                }
            } else {
            // one unit = 32 channels of one output row for this lane's pixel
            auto unit = [&](int t, int c0, float (&v)[32]) {
                const uint32_t t_row = tmem_base + (uint32_t)((acc * p.R + (p.stack ? p.R - 1 - t : t)) * p.acc_stride) + ((uint32_t)(q * 32) << 16);
                tmem_ld32(t_row + c0, v);
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const float4 sc = *reinterpret_cast<const float4*>(&s_scale[c0 + j]);
                    const float4 sh = *reinterpret_cast<const float4*>(&s_shift[c0 + j]);
                    v[j]     = fmaxf(fmaf(v[j],     sc.x, sh.x), lower);
                    v[j + 1] = fmaxf(fmaf(v[j + 1], sc.y, sh.y), lower);
                    v[j + 2] = fmaxf(fmaf(v[j + 2], sc.z, sh.z), lower);
                    v[j + 3] = fmaxf(fmaf(v[j + 3], sc.w, sh.w), lower);
                }
            };
            if (PLANAR) {
                // last conv of a FastDVDnet DenBlock: the NPL real channels leave as planar frames, residual form
                // in1 - net (models.py:196) applied here; lanes are consecutive pixels -> coalesced plane accesses
#pragma unroll
                for (int i = 0; i < PIN_ROWS; ++i) {
                    const int t = g + i * EPI_WG;
                    if (t < rows) {
                        float v[32];
                        unit(t, 0, v);
                        if (valid) {
                            const long o = (long)n * NPL * pl_plane + (long)(y0 + t) * p.W + wo;
#pragma unroll
                            for (int c = 0; c < NPL; ++c) p.planar_out[o + c * pl_plane] = pin[i][c] - v[c];
                        }
                    }
                }
            } else {
                for (int u = g; u < units; u += EPI_WG) {
                    const int t = u / nch, c0 = (u - t * nch) << 5;
                    const int ho = y0 + t;
                    float v[32];
                    if (MODE == 4 || MODE == 5) {
                        // ---- data gradient + activation backward, fused (replaces a separate pass over dy, y and dz) ----
                        // operands of this unit from global memory first (the other warpgroup hides their latency)
                        float4 yy[8], ra[8];
                        const long eo = out_offset(ho, c0);
#pragma unroll
                        for (int j = 0; j < 8; ++j) { yy[j] = make_float4(0.f, 0.f, 0.f, 0.f); ra[j] = yy[j]; }
                        if (valid) {
                            const float4* yp = reinterpret_cast<const float4*>(p.mask_y + eo);
#pragma unroll
                            for (int j = 0; j < 8; ++j) yy[j] = __ldg(yp + j);
                            if (p.residual) {
                                const float4* rp = reinterpret_cast<const float4*>(p.residual + eo);
#pragma unroll
                                for (int j = 0; j < 8; ++j) ra[j] = __ldg(rp + j);
                            }
                        }
                        unit(t, c0, v);
                        const uint32_t sbuf = sbuf0;
                        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // previous store has read the tile
                        __syncwarp();
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const float ya[4] = {yy[j].x, yy[j].y, yy[j].z, yy[j].w};
                            const float rv[4] = {ra[j].x, ra[j].y, ra[j].z, ra[j].w};
                            float pz[4];
#pragma unroll
                            for (int e = 0; e < 4; ++e) {
                                float d = v[4 * j + e] + rv[e];
                                if (p.round_tf32) d = rna_tf32(d);
                                if (!valid || (p.mask_relu && !(ya[e] > 0.f))) d = 0.f;
                                v[4 * j + e] = d;
                                pz[e] = d * ya[e];
                            }
                            // phase 1: dz * y into the staging tile (column sums for the BatchNorm scale gradient)
                            const uint32_t a = sbuf + (uint32_t)lane * 128u + (uint32_t)((j ^ (lane & 7)) << 4);
                            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(pz[0]), "f"(pz[1]), "f"(pz[2]), "f"(pz[3]) : "memory");
                        }
                        __syncwarp();
                        // lane c sums column c of the 32 x 32 tile: element (row r, column c) sits in chunk (c >> 2) ^ (r & 7) of
                        // row r - for a fixed r the 32 lanes hit 32 different banks
                        float cs2 = 0.f;
                        if (p.col_s2) {
#pragma unroll 8
                            for (int r = 0; r < 32; ++r) {
                                float e;
                                const uint32_t a = sbuf + (uint32_t)r * 128u + (uint32_t)((((lane >> 2) ^ (r & 7)) << 4) + ((lane & 3) << 2));
                                asm volatile("ld.shared.f32 %0, [%1];" : "=f"(e) : "r"(a) : "memory");
                                cs2 += e;
                            }
                        }
                        __syncwarp();
                        // phase 2: dz itself -> column sums (bias / BatchNorm shift gradient) and the TMA store
#pragma unroll
                        for (int j = 0; j < 32; j += 4) {
                            const uint32_t a = sbuf + (uint32_t)lane * 128u + (uint32_t)(((j >> 2) ^ (lane & 7)) << 4);
                            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v[j]), "f"(v[j + 1]), "f"(v[j + 2]), "f"(v[j + 3]) : "memory");
                        }
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        __syncwarp();
                        if (lane == 0) {
                            const int cg = p.col0 + c0;
                            int cx = cg, cw = wt * 128 + q * 32, chh = ho;
                            if (p.ps) { const int qq = cg / Cq; cx = cg % Cq; cw = 2 * cw + (qq & 1); chh = 2 * ho + (qq >> 1); }
                            asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                                         ::"l"(&tmY), "r"(sbuf), "r"(cx), "r"(cw), "r"(chh), "r"(n) : "memory");
                            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                        }
                        if (p.col_s1) {
                            float cs1 = 0.f;
#pragma unroll 8
                            for (int r = 0; r < 32; ++r) {
                                float e;
                                const uint32_t a = sbuf + (uint32_t)r * 128u + (uint32_t)((((lane >> 2) ^ (r & 7)) << 4) + ((lane & 3) << 2));
                                asm volatile("ld.shared.f32 %0, [%1];" : "=f"(e) : "r"(a) : "memory");
                                cs1 += e;
                            }
                            // column of the stored tensor this lane summed (PixelShuffle: the sub-pixel groups share the channels)
                            const int cg = p.col0 + c0;
                            const int cc = (p.ps ? cg % Cq : cg) + lane;
                            if (MODE == 5) {
                                // this warp's own row of partials: every address has ONE writer (lane cc % 32 of this warp)
                                // and a thread's reductions to one address apply in program order, i.e. in the fixed order
                                // the units reach the warp - the fire-and-forget shared reduction of MODE 4, deterministic
                                atomicAdd(&s_wcs[warp - 4][0][cc], cs1);
                                if (p.col_s2) atomicAdd(&s_wcs[warp - 4][1][cc], cs2);
                            } else {
                                atomicAdd(&s_cs1[cc], cs1);
                                if (p.col_s2) atomicAdd(&s_cs2[cc], cs2);
                            }
                        }
                        __syncwarp();
                        continue;
                    }
                    unit(t, c0, v);
                    if (MODE == 1) {
                        float4 rn[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) rn[j] = make_float4(0.f, 0.f, 0.f, 0.f);
                        const int un = u + EPI_WG;
                        if (p.residual && valid && un < units) {          // prefetch the skip values of this warp's next unit
                            const int tn = un / nch;
                            const float4* rp = reinterpret_cast<const float4*>(p.residual + out_offset(y0 + tn, (un - tn * nch) << 5));
#pragma unroll
                            for (int j = 0; j < 8; ++j) rn[j] = __ldg(rp + j);
                        }
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            v[4 * j] += rr[j].x; v[4 * j + 1] += rr[j].y; v[4 * j + 2] += rr[j].z; v[4 * j + 3] += rr[j].w;
                            rr[j] = rn[j];
                        }
                    }
                    if (p.round_tf32) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) v[j] = rna_tf32(v[j]);
                    }
                    // coalesced path: the warp's 32 pixels x 32 channels go through a 128B-swizzled 4 KB staging tile and
                    // leave as ONE TMA store (box {32 ch, 32 px}; PixelShuffle = element stride 2 on the pixel axis of a map
                    // over the up-sampled tensor); out-of-image pixels are clipped by TMA
                    const uint32_t sbuf = sbuf0 + (p.out_bufs == 2 ? (st_cnt & 1) * tile_b : 0u);
                    if (lane == 0) {
                        if (p.out_bufs == 2) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
                        else                 asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                    }
                    __syncwarp();
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        const uint32_t a = sbuf + (uint32_t)lane * 128u + (uint32_t)(((j >> 2) ^ (lane & 7)) << 4);
                        asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v[j]), "f"(v[j + 1]), "f"(v[j + 2]), "f"(v[j + 3]) : "memory");
                    }
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) {
                        const int cg = p.col0 + c0;
                        int cx = cg, cw = wt * 128 + q * 32, chh = ho;
                        if (p.ps) { const int qq = cg / Cq; cx = cg % Cq; cw = 2 * cw + (qq & 1); chh = 2 * ho + (qq >> 1); }
                        asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                                     ::"l"(&tmY), "r"(sbuf), "r"(cx), "r"(cw), "r"(chh), "r"(n) : "memory");
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    }
                    ++st_cnt;
                }
            }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty_bar[acc]);
            if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
        }
        if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");    // TMA stores (if any) have landed
        if (MODE == 4 && p.col_s1) {
            // all epilogue warps of the CTA have added their partial sums: one global atomic per column and CTA
            asm volatile("bar.sync 1, %0;" ::"r"(128 * EPI_WG) : "memory");
            const int e = threadIdx.x - 128;
            const int ncol = p.ps ? Cq : p.Ctot;
            if (e < min(ncol, 128)) {
                atomicAdd(p.col_s1 + e, s_cs1[e]);
                if (p.col_s2) atomicAdd(p.col_s2 + e, s_cs2[e]);
            }
        }
        if (MODE == 5 && p.col_s1) {
            // column e of the CTA's slot = the epilogue warps' partials added in warp order
            asm volatile("bar.sync 1, %0;" ::"r"(128 * EPI_WG) : "memory");
            const int e = threadIdx.x - 128;
            const int ncol = p.ps ? Cq : p.Ctot;
            if (e < min(ncol, 128)) {
                float a1 = s_wcs[0][0][e], a2 = s_wcs[0][1][e];
#pragma unroll
                for (int w = 1; w < 4 * EPI_WG; ++w) { a1 += s_wcs[w][0][e]; a2 += s_wcs[w][1][e]; }
                float* slot = p.col_s1 + (long)blockIdx.x * 2 * ncol;
                slot[e] = a1;
                if (p.col_s2) slot[ncol + e] = a2;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------------
// host side: TMA descriptors through the driver entry point (no libcuda link dependency), launches
// ---------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// cuTensorMapEncodeTiled of a rank-`rank` fp32 / fp16 tensor: dims, box and element strides innermost first, byte strides
// of dims 1 .. rank-1.  `what` names the tensor in the error message.
int encode_map(CUtensorMap* tm, const char* what, const void* base, bool half, int rank, const cuuint64_t* dims,
               const cuuint64_t* strides, const cuuint32_t* box, const cuuint32_t* estr, CUtensorMapSwizzle swz,
               CUtensorMapL2promotion l2 = CU_TENSOR_MAP_L2_PROMOTION_L2_256B) {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    if (!fn) return sci_fail(SCI_ELAUNCH, "cuTensorMapEncodeTiled entry point not available");
    const CUresult r = fn(tm, half ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (cuuint32_t)rank,
                          const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz, l2,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        char msg[96];
        snprintf(msg, sizeof(msg), "cuTensorMapEncodeTiled(%s) failed with CUresult %d", what, (int)r);
        return sci_fail(SCI_ELAUNCH, msg);
    }
    return SCI_OK;
}

// NHWC activation tensor [N][H][W][C], box = {32 ch, box_w*stride, box_h*stride, 1} traversed with element stride `stride`
int make_act_map(CUtensorMap* tm, const float* x, int N, int H, int W, int C, int stride, int box_w, int box_h,
                 CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B, bool half = false, bool row64 = false) {
    const cuuint64_t esz = half ? 2 : 4;
    const cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
    const cuuint64_t strides[3] = {(cuuint64_t)C * esz, (cuuint64_t)W * C * esz, (cuuint64_t)H * W * C * esz};
    const cuuint32_t box[4] = {(cuuint32_t)(row64 ? 32 : (half ? 64 : KCH)), (cuuint32_t)(box_w * stride), (cuuint32_t)(box_h * stride), 1};
    const cuuint32_t estr[4] = {1, (cuuint32_t)stride, (cuuint32_t)stride, 1};
    return encode_map(tm, "activations", x, half, 4, dims, strides, box, estr, swz);
}

// packed weights [taps][Cout][Cin] (taps = 9, or 18 with the hi/remainder split), box = {32 ch, Cout, 1}
int make_weight_map(CUtensorMap* tm, const float* w, int Cout, int Cin, int taps, int box_rows = 0, bool half = false,
                    bool row64 = false) {
    const cuuint64_t esz = half ? 2 : 4;
    const cuuint64_t dims[3] = {(cuuint64_t)Cin, (cuuint64_t)Cout, (cuuint64_t)taps};
    const cuuint64_t strides[2] = {(cuuint64_t)Cin * esz, (cuuint64_t)Cout * Cin * esz};
    const cuuint32_t box[3] = {(cuuint32_t)(row64 ? 32 : (half ? 64 : KCH)), (cuuint32_t)(box_rows ? box_rows : Cout), 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    return encode_map(tm, "weights", w, half, 3, dims, strides, box, estr,
                      row64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B);
}

// Launches `kernel` with up to 220 KB of dynamic shared memory.  pdl: with programmatic stream serialization, so that
// its prologue may overlap the tail of the previous kernel on the stream (the kernel waits with griddepcontrol.wait
// before it reads that kernel's results).
template <typename... Params, typename... Args>
int launch(void (*kernel)(Params...), dim3 grid, int threads, size_t smem, void* stream, bool pdl, const char* what,
           const Args&... args) {
    cudaError_t e = sci_smem_limit((const void*)kernel, 220 * 1024);
    if (e != cudaSuccess) return sci_fail(SCI_ELAUNCH, what, e);
    if (pdl) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = grid; cfg.blockDim = dim3(threads); cfg.dynamicSmemBytes = smem; cfg.stream = sci_stream(stream);
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        e = cudaLaunchKernelEx(&cfg, kernel, args...);
    } else {
        kernel<<<grid, threads, smem, sci_stream(stream)>>>(args...);
        e = cudaGetLastError();
    }
    return e == cudaSuccess ? SCI_OK : sci_fail(SCI_ELAUNCH, what, e);
}

int next_pow2_cols(int c) { int v = 32; while (v < c) v <<= 1; return v; }

int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return v ? atoi(v) : dflt;
}

// bytes per operand row: fp16 tensors with 32 channels use 64-byte rows (SWIZZLE_64B); everything else one 128-byte row
// per pixel and channel chunk
int operand_row_bytes(const sci_conv_desc* d) {
    return (d->half_io && d->Cin == 32 && env_int("SCI_CONV_SW64", 1)) ? 64 : 128;
}

// K steps (32 bytes: 8 fp32 / 16 fp16 channels each) of the LAST channel chunk that can hold non-zero channels when only
// the first `used` of the Cin channels can: the zero-padded rest is not multiplied.  `used` must reach into the last chunk
// to shorten it.
int ks_last(int Cin, int used, int rb_in, int esz) {
    const int kch = rb_in / esz, step = 32 / esz, rest = used - (Cin / kch - 1) * kch;
    return rest <= 0 ? rb_in / 32 : min(rb_in / 32, (rest + step - 1) / step);
}

int conv_fwd_tc_launch(const sci_conv_desc* d, void* stream) {
    const bool half = d->half_io != 0;
    const int esz = half ? 2 : 4;
    const int rb_in = operand_row_bytes(d);
    const int kch = rb_in / esz;
    if (d->Cin % kch != 0 || d->Cout % 16 != 0 || d->Cout > 256)
        return sci_fail(SCI_EUNSUPPORTED, "conv tc: needs Cin % 32 == 0 (fp16: % 64), Cout % 16 == 0, Cout <= 256");
    if (((uintptr_t)d->x | (uintptr_t)d->w | (uintptr_t)d->y | (uintptr_t)d->residual) & 15)
        return sci_fail(SCI_EINVAL, "conv tc: pointers must be 16-byte aligned");
    if (d->pixel_shuffle && (d->Cout % 128 != 0))
        return sci_fail(SCI_EUNSUPPORTED, "conv tc: pixel_shuffle needs Cout % 128 == 0");
    if (half && (d->pixel_shuffle || d->residual || d->w_split || d->emit_lo || d->Cout % 32))
        return sci_fail(SCI_EUNSUPPORTED, "conv tc fp16 (tile kernel): plain layers with Cout % 32 == 0 only");
    FwdParams p;
    p.scale = d->scale; p.shift = d->shift; p.residual = d->residual; p.y = d->y;
    p.N = d->N; p.H = d->H; p.W = d->W; p.stride = d->stride;
    p.Ho = (d->H - 1) / d->stride + 1; p.Wo = (d->W - 1) / d->stride + 1;
    p.Cin = d->Cin; p.Cout = d->Cout; p.relu = d->relu; p.ps = d->pixel_shuffle; p.round_tf32 = d->round_tf32;
    p.wsplit = d->w_split ? 1 : 0;
    p.emit_lo = d->emit_lo ? 1 : 0;
    p.Cstore = (half && d->Cout_store) ? d->Cout_store : d->Cout;
    p.ks_last = ks_last(d->Cin, (d->K_used > 0 && d->K_used <= d->Cin && !d->w_split) ? d->K_used : d->Cin, rb_in, esz);
    if (p.emit_lo && (d->pixel_shuffle || d->residual || !d->round_tf32))
        return sci_fail(SCI_EUNSUPPORTED, "conv tc: emit_lo needs round_tf32 and no pixel_shuffle / residual");
    p.tiles_w = (p.Wo + TILE_W - 1) / TILE_W; p.tiles_h = (p.Ho + TILE_H - 1) / TILE_H;
    p.num_tiles = p.tiles_w * p.tiles_h * p.N;
    p.k_chunks = p.Cin / kch;
    p.rb_in = rb_in;
    p.a_bytes = TILE_W * TILE_H * rb_in;
    int stage_bytes = p.a_bytes + p.Cout * rb_in * (1 + p.wsplit);
    // (fp16 chains only: the fp32 training layers measured 76 -> 81 us with three 72 KB stages instead of eight of 24 KB)
    p.tps = (half && (216 * 1024) / (3 * stage_bytes) >= 3 && env_int("SCI_CONV_TPS", 3) == 3) ? 3 : 1;
    stage_bytes *= p.tps;
    p.stages = min(MAX_STAGES, (216 * 1024) / stage_bytes);
    p.acc_stride = ((p.Cout + 31) / 32) * 32;
    p.lo_chunk0 = 0;
    if (p.wsplit && !half && d->lo_channel0 > 0 && d->lo_channel0 % KCH == 0 && d->lo_channel0 < d->Cin && 4 * p.acc_stride <= 512 &&
        env_int("SCI_CONV_SPLIT_ACC", 1)) {
        p.lo_chunk0 = d->lo_channel0 / KCH;
        p.acc_stride *= 2;                               // [main | small products] per accumulator buffer
    }
    p.tmem_cols = next_pow2_cols(2 * p.acc_stride);
    CUtensorMap tmA, tmB;
    const int cin_store = (half && d->Cin_store) ? d->Cin_store : d->Cin;
    int rc = make_act_map(&tmA, d->x, d->N, d->H, d->W, cin_store, d->stride, TILE_W, TILE_H,
                          rb_in == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B, half, rb_in == 64);
    if (rc) return rc;
    rc = make_weight_map(&tmB, d->w, d->Cout, d->Cin, 9 * (1 + p.wsplit), 0, half, rb_in == 64);
    if (rc) return rc;
    const size_t smem = (size_t)p.stages * stage_bytes + 1024;
    const int grid = min(p.num_tiles, SCI_NUM_SMS);
    p.pdl = (d->pdl && env_int("SCI_CONV_PDL", 1)) ? 1 : 0;
    if (env_int("SCI_CONV_VERBOSE", 0))
        fprintf(stderr, "conv v1 plan: %dx%d Cin %d -> %d stride %d half %d ps %d | tps %d stages %d lo_chunk0 %d ks_last %d wsplit %d "
                "emit_lo %d pdl %d tiles %d\n", d->H, d->W, d->Cin, d->Cout, d->stride, (int)half, p.ps, p.tps, p.stages, p.lo_chunk0,
                p.ks_last, p.wsplit, p.emit_lo, p.pdl, p.num_tiles);
    return launch(half ? conv_fwd_tc_kernel<true> : conv_fwd_tc_kernel<false>, dim3(grid), TC_THREADS, smem, stream, p.pdl,
                  "conv tc fwd", tmA, tmB, p);
}




bool fwd2_eligible(const sci_conv_desc* d) {
    if (d->planar_out) return true;                      // fused planar output exists in the v2 kernel only
    if (d->half_io) return d->stride == 1;
    return d->stride == 1 && d->Cout % 32 == 0 && (d->Cout <= 128 || d->Cout == 256) && !d->w_split && !d->emit_lo &&
           env_int("SCI_CONV_V2", 1) != 0;
}

// columns [col0, col0 + ncols) of the layer.  ord_slots != NULL: fused data gradient with fixed-order column sums (MODE 5)
// into the [grid][2][stored channels] slots there.  grid_out: the launch's grid; plan_only: only that, no launch.
int conv_fwd2_tc_launch(const sci_conv_desc* d, void* stream, int col0, int ncols, float* ord_slots = nullptr,
                        int* grid_out = nullptr, bool plan_only = false) {
    const bool half = d->half_io != 0;
    const int esz = half ? 2 : 4;
    const int rb_in = operand_row_bytes(d);
    const int kch = rb_in / esz;                     // channels per operand row
    if (d->Cin % kch != 0) return sci_fail(SCI_EUNSUPPORTED, "conv tc v2: Cin % 32 (fp32) / % 64 or == 32 (fp16)");
    if (((uintptr_t)d->x | (uintptr_t)d->w | (uintptr_t)d->y | (uintptr_t)d->residual) & 15)
        return sci_fail(SCI_EINVAL, "conv tc: pointers must be 16-byte aligned");
    const int cin_store = (half && d->Cin_store) ? d->Cin_store : d->Cin;       // channels per pixel of the stored input
    const int cout_store = (half && d->Cout_store) ? d->Cout_store : (d->pixel_shuffle ? d->Cout / 4 : d->Cout);
    if (half && (cin_store % 8 || cout_store % 8 || cin_store > d->Cin))
        return sci_fail(SCI_EINVAL, "conv tc v2 fp16: stored channel counts must be multiples of 8 (16-byte TMA strides)");
    Fwd2Params p;
    p.scale = d->scale; p.shift = d->shift; p.residual = d->residual; p.y = d->y;
    p.N = d->N; p.H = d->H; p.W = d->W; p.Cin = d->Cin; p.Cout = ncols; p.col0 = col0; p.Ctot = d->Cout;
    p.relu = d->relu; p.ps = d->pixel_shuffle; p.round_tf32 = d->round_tf32;
    p.planar_in1 = d->planar_in1; p.planar_out = d->planar_out;
    if (p.planar_out && (!p.planar_in1 || p.ps || p.Cout != 32 || d->residual))
        return sci_fail(SCI_EINVAL, "conv tc v2: planar output needs planar_in1, Cout == 32, no pixel_shuffle / residual");
    p.tiles_w = (p.W + 127) / 128;
    p.k_chunks = p.Cin / kch;
    const int rb_out = (half && cout_store == 32 && !p.planar_out) ? 64 : 128;
    p.rb_in = rb_in; p.rb_out = rb_out;
    p.a_stage = rb_in == 64 ? 9 * 1024 : A2_STAGE;
    p.row_bytes = ROW_PX * rb_in;
    p.desc_hi = rb_in == 64 ? DESC_HI_K64 : DESC_HI_K128;
    const int a_stage = p.a_stage;
    const int b_bytes = p.Cout * rb_in;
    const bool tma_store = !p.planar_out;            // every epilogue but the planar one leaves through TMA stores
    p.Cstore = cout_store;
    p.ks_last = ks_last(d->Cin, (d->K_used > 0 && d->K_used <= d->Cin) ? d->K_used : d->Cin, rb_in, esz);
    p.ucols = 32;
    if (half) {
        const int cq = p.ps ? d->Cout / 4 : ncols;             // columns that belong to one stored pixel row
        if (cq % 32 != 0) return sci_fail(SCI_EUNSUPPORTED, "conv tc v2 fp16: column groups of 32");
        p.ucols = (cq % 64 == 0 || cq > 64) ? 64 : 32;
        if (rb_out == 64 && p.ucols != 32) return sci_fail(SCI_EUNSUPPORTED, "conv tc v2 fp16: a 32-channel output tensor needs 32-column units");
        if (p.ps && cq != 32 && cq % 64 != 0) return sci_fail(SCI_EUNSUPPORTED, "conv tc v2 fp16: PixelShuffle groups of 32 or k*64 columns");
    }
    p.split = 0;
    if (half && d->w_split) {
        // fp16 value + remainder form (FFDNet inference): d->Cin = 64 * (groups of 32 real input channels), stored output = 2 * Cout
        if (rb_in != 128 || p.ps || d->residual || p.planar_out || ncols != d->Cout || d->Cout % 32 || d->Cout > 128 || cout_store != 2 * d->Cout)
            return sci_fail(SCI_EUNSUPPORTED, "conv tc v2 fp16 split: plain layers, Cout % 32 == 0, Cout <= 128, Cout_store == 2 * Cout");
        p.split = (d->K_used > 0 && d->K_used <= 16 && p.k_chunks == 1) ? 1 : 2;
        p.ucols = 32;
        p.ks_last = 4;
    }
    int mode = p.planar_out ? (d->planar_planes == 1 ? 3 : 2) : (d->residual ? 1 : 0);
    p.mask_y = d->mask_y; p.col_s1 = d->col_s1; p.col_s2 = d->col_s2; p.mask_relu = d->mask_relu;
    if (d->mask_y) {
        if (half || p.planar_out || (d->pixel_shuffle ? d->Cout / 4 : d->Cout) > 128 || (d->col_s2 && !d->col_s1))
            return sci_fail(SCI_EUNSUPPORTED, "conv tc v2: fused activation backward needs the fp32 TMA-store path and <= 128 stored channels");
        mode = 4;
        if (ord_slots && d->col_s1) { mode = 5; p.col_s1 = ord_slots; }
    }
    const int w_bytes = 9 * p.k_chunks * b_bytes;
    // shared-memory plan: [resident weights] [pipeline stages] [store staging: 4 * epi_wg warps x out_bufs x 4 KB].
    // Two epilogue warpgroups (see the kernel comment) unless their extra staging would cost the weights their residency.
    const int total_budget = 214 * 1024;
    const int tile_b = 32 * rb_out;                   // staging tile of one epilogue warp (fp32 path: rb_out = 128)
    int out_stage = 0, budget = 0, epi_wg = 2;
    const int epi_env = env_int("SCI_CONV_EPI_WG", 0);
    // measured per layer (tools/pass_layers.py): the second warpgroup pays where the epilogue work per MMA is high (K <= 32:
    // 12->90 0.270 -> 0.255 ms, or a skip-add: 64->128+PS 0.251 -> 0.178 ms) and costs where the MMA-issuing warp is the
    // critical path and now shares its scheduler with two epilogue warps (128->128: 0.067 -> 0.078 ms)
    const int epi_first = epi_env ? (epi_env == 1 ? 1 : 2) : ((half || p.k_chunks <= 1 || d->residual || d->mask_y) ? 2 : 1);
    for (epi_wg = epi_first; epi_wg >= 1; --epi_wg) {
        for (p.out_bufs = ((epi_wg == 2 || d->mask_y) ? 1 : 2); p.out_bufs >= 1; --p.out_bufs) {
            out_stage = tma_store ? 4 * epi_wg * p.out_bufs * tile_b : 0;
            budget = total_budget - out_stage;
            p.resident = (w_bytes + 3 * a_stage <= budget) ? 1 : 0;
            const int sb = a_stage + (p.resident ? 0 : 3 * b_bytes);
            const int st = (budget - (p.resident ? w_bytes : 0)) / sb;
            const bool would_be_resident = w_bytes + 3 * a_stage <= total_budget - (tma_store ? 4 * epi_wg * tile_b : 0);
            if ((p.resident || !would_be_resident) && st >= 3) break;
            if (p.out_bufs == 1) break;
        }
        const bool resident_with_one = w_bytes + 3 * a_stage <= total_budget - (tma_store ? 4 * tile_b : 0);
        // fp16 chains: the MMAs are twice as fast, so the epilogue decides more often - two warpgroups even where that costs
        // the weights their residency (64->128 + PixelShuffle: 0.215 ms resident with one group, 0.135 ms streamed with two)
        if (epi_wg == 1 || epi_env == 2 || half || p.resident || !resident_with_one) break;
    }
    if (env_int("SCI_CONV_RESIDENT", 1) == 0) p.resident = 0;
    int stage_bytes = a_stage + (p.resident ? 0 : 3 * b_bytes);
    p.stages = min(MAX_STAGES, (budget - (p.resident ? w_bytes : 0)) / stage_bytes);
    if (p.stages < 2) return sci_fail(SCI_EUNSUPPORTED, "conv tc v2: pipeline does not fit");
    p.acc_stride = p.split ? 2 * p.Cout : p.Cout;        // split: [main | value x remainder products]
    if (p.split && 2 * p.acc_stride > 512) return sci_fail(SCI_EUNSUPPORTED, "conv tc v2 fp16 split: accumulators do not fit");
    // super-tiles of R output rows: the R+2 input rows are loaded once and feed up to three output rows each, which
    // cuts the shared-memory fill traffic per output row from 3 rows to (R+2)/R.  Measured (tools/bench_conv.py): the
    // resident-weight layers are bound by ring_bytes / load round-trip latency, i.e. by bytes per output tile.
    // R accumulators x 2 buffers must fit the 512 TMEM columns; streamed weights keep R = 1 (their B tiles are per filter row).
    p.R = 1;
    if (!p.resident && !p.split && 2 * 2 * p.acc_stride <= 512 && p.H >= 2 && env_int("SCI_CONV_WPAIR", 1)) {
        // streamed weights: two output rows per tile share every weight tile (a stage then carries two input rows)
        // ... where the image is large enough that halving the tile count does not cost a wave of the 148 persistent CTAs
        // (8x128x128: 1024 one-row tiles = 6.9 waves; 512 two-row tiles would be 3.5 -> 4 waves of twice the work)
        const int sb2 = 2 * a_stage + 3 * b_bytes;
        const long tiles2 = (long)p.tiles_w * ((p.H + 1) / 2) * p.N;
        if (budget / sb2 >= 2 && tiles2 >= 8L * SCI_NUM_SMS) p.R = 2;
    }
    if (p.resident && !p.split) {             // (the split issuer is written for one output row per tile)
        const int rmax = env_int("SCI_CONV_ROWS", 8);
        while (p.R * 2 <= rmax && 2 * (p.R * 2) * p.acc_stride <= 512 && p.R * 2 <= p.H) p.R *= 2;
    }
    if (!p.resident && p.R == 2) {
        stage_bytes = 2 * a_stage + 3 * b_bytes;
        p.stages = min(MAX_STAGES, budget / stage_bytes);
    }
    p.stack = (p.resident && p.R >= 2 && 3 * p.Cout <= 256 && env_int("SCI_CONV_STACK", 1)) ? 1 : 0;
    p.tiles_h = (p.H + p.R - 1) / p.R;
    p.num_tiles = p.tiles_w * p.tiles_h * p.N;
    p.tmem_cols = next_pow2_cols(2 * p.R * p.acc_stride);
    p.dbg = env_int("SCI_CONV_DBG", 0);
    const int grid = min(p.num_tiles, SCI_NUM_SMS);
    if (grid_out) *grid_out = grid;
    if (plan_only) return SCI_OK;
    CUtensorMap tmA, tmB;
    // activation map with a {kch ch, 130 px, 1 row, 1 image} box.  fp16: the channel extent is the STORED one; a box that
    // sticks out of it (e.g. channels 64..127 of a 96-channel tensor) is zero-filled by TMA, matching the zero rows of the
    // packed weights
    int rc = make_act_map(&tmA, d->x, d->N, d->H, d->W, cin_store, 1, ROW_PX, 1,
                          rb_in == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B, half, rb_in == 64);
    if (rc) return rc;
    rc = make_weight_map(&tmB, d->w, d->Cout, d->Cin, 9, ncols, half, rb_in == 64);
    if (rc) return rc;
    CUtensorMap tmY = tmA;
    if (tma_store) {
        // plain layers: [N][H][W][Cout], box {32 ch, 32 px}.  PixelShuffle layers: the map covers the up-sampled tensor
        // [N][2H][2W][Cout/4]; the 32 pixels of a warp land on every second column (element stride 2).
        const int ps = d->pixel_shuffle ? 1 : 0;
        const cuuint64_t oc = (cuuint64_t)cout_store, ow = (cuuint64_t)(d->W << ps), oh = (cuuint64_t)(d->H << ps);
        const cuuint64_t dims[4] = {oc, ow, oh, (cuuint64_t)d->N};
        const cuuint64_t strides[3] = {oc * esz, ow * oc * esz, oh * ow * oc * esz};
        const cuuint32_t box[4] = {(cuuint32_t)(rb_out / esz), (cuuint32_t)(32 << ps), 1, 1};
        const cuuint32_t estr[4] = {1, (cuuint32_t)(1 << ps), 1, 1};
        rc = encode_map(&tmY, "output", d->y, half, 4, dims, strides, box, estr,
                        rb_out == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE);
        if (rc) return rc;
    }
    const size_t smem = (size_t)(p.resident ? w_bytes : 0) + (size_t)p.stages * stage_bytes + out_stage + 1024;
    if (smem > 220 * 1024) return sci_fail(SCI_EUNSUPPORTED, "conv tc v2: shared memory budget exceeded");
    typedef void (*Fwd2Kernel)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const Fwd2Params);
    // indexed by MODE (MODEs 4 and 5 exist for fp32 only)
    static const Fwd2Kernel kernels[2][2][6] = {
        {{conv_fwd2_tc_kernel<1, 0, false>, conv_fwd2_tc_kernel<1, 1, false>, conv_fwd2_tc_kernel<1, 2, false>,
          conv_fwd2_tc_kernel<1, 3, false>, conv_fwd2_tc_kernel<1, 4, false>, conv_fwd2_tc_kernel<1, 5, false>},
         {conv_fwd2_tc_kernel<2, 0, false>, conv_fwd2_tc_kernel<2, 1, false>, conv_fwd2_tc_kernel<2, 2, false>,
          conv_fwd2_tc_kernel<2, 3, false>, conv_fwd2_tc_kernel<2, 4, false>, conv_fwd2_tc_kernel<2, 5, false>}},
        {{conv_fwd2_tc_kernel<1, 0, true>, conv_fwd2_tc_kernel<1, 1, true>, conv_fwd2_tc_kernel<1, 2, true>,
          conv_fwd2_tc_kernel<1, 3, true>, nullptr, nullptr},
         {conv_fwd2_tc_kernel<2, 0, true>, conv_fwd2_tc_kernel<2, 1, true>, conv_fwd2_tc_kernel<2, 2, true>,
          conv_fwd2_tc_kernel<2, 3, true>, nullptr, nullptr}}};
    const Fwd2Kernel kern = kernels[half ? 1 : 0][epi_wg - 1][mode];
    if (!kern) return sci_fail(SCI_EUNSUPPORTED, "conv tc v2: epilogue not built");
    const int threads = 128 + 128 * epi_wg;
    p.pdl = (d->pdl && env_int("SCI_CONV_PDL", 1)) ? 1 : 0;
    if (env_int("SCI_CONV_VERBOSE", 0))
        fprintf(stderr, "conv v2 plan: %dx%d Cin %d -> %d cols (+%d) half %d ps %d mode %d | resident %d stages %d R %d stack %d epi_wg %d out_bufs %d "
                "rb %d/%d smem %zu KB tiles %d split %d ks_last %d pdl %d\n", d->H, d->W, d->Cin, ncols, col0, (int)half, p.ps, mode, p.resident,
                p.stages, p.R, p.stack, epi_wg, p.out_bufs, rb_in, rb_out, smem / 1024, p.num_tiles, p.split, p.ks_last, p.pdl);
    return launch(kern, dim3(grid), threads, smem, stream, p.pdl, "conv tc fwd v2", tmA, tmB, tmY, p);
}

// ---------------------------------------------------------------------------------------------------
// weight-gradient kernel, version 2 (conv_wgrad2_tc_kernel): operand orientation and tap fusion chosen per layer
//   dW[tap][co][ci] += oscale[co] * sum_pixels dz[p][co] * x[p (+) tap][ci]
//   GEMM view: D[128][N] += A^T B over K = pixels, both operands MN-major (channels contiguous; TMA swizzle
//   128B_ATOM_32B <-> UMMA SWIZZLE_128B_BASE32B, the only MN-major layout tcgen05 accepts for TF32), built from TMA boxes
//   {32 ch, 8 px, 8 rows, 1 image} of dz and of x at the tap-shifted (and, for stride-2 layers, element-strided)
//   coordinates; out-of-image pixels are zero-filled.  One CTA group owns a filter row and one 128-wide M block, each
//   CTA a strided subset of the 8x8 pixel tiles; it accumulates in TMEM and finishes with red.global.add into the
//   packed gradient (ORDERED: with plain stores into its own region of slot blockIdx.x of a [gx][9][Cout][Cin] workspace
//   at p.dw, which sci_ordered_slot_sum adds into dw in slot order).  The launch list of a first version with M = Cout fixed (profiles/) showed the full-resolution
//   32-channel layers at 0.73-0.89 ms each: with M = 32 of 128 rows used, three quarters of every MMA were wasted and
//   each tap reloaded the dz tile.  Hence
//   * swap = 0: M side = dz (Cout), N side = x.  swap = 1: M side = x (Cin), N side = dz (Cout) - chosen when that
//     fills the 128 MMA rows better.
//   * fuse = 1: the three horizontal taps of the filter row are ONE operand (their 32-channel chunks are simply
//     consecutive chunks of the MN-major operand), so one MMA per 8 pixels covers all three taps and the unshifted
//     operand is loaded once per tile instead of once per tap.
// ---------------------------------------------------------------------------------------------------
constexpr int WG_TILE = 8;                       // 8x8 pixels = 64 = K block
constexpr int WG_CHUNK_BYTES = WG_TILE * WG_TILE * KCH * 4;   // 8 KB per 32-channel chunk

struct Wgrad2Params {
    const float* oscale; float* dw;
    int N, Ho, Wo, Cin, Cout, stride;
    int tiles_w, tiles_h, num_tiles;
    int swap, fuse, p_chunks, q_chunks, n_mma, accs, m_tiles, tmem_cols, stages;
};

template <bool ORDERED>
__global__ void __launch_bounds__(TC_THREADS, 1)
conv_wgrad2_tc_kernel(const __grid_constant__ CUtensorMap tmZ, const __grid_constant__ CUtensorMap tmX, const Wgrad2Params p) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[4], empty_bar[4], done_bar;
    __shared__ uint32_t tmem_slot;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const int frow = blockIdx.y / p.m_tiles, mt = blockIdx.y % p.m_tiles;
    const int cin_chunks = p.Cin / KCH, cout_chunks = p.Cout / KCH;
    const int p_chunks = p.swap ? p.p_chunks : min(cout_chunks - mt * 4, 4);
    const uint32_t p_region = 4 * WG_CHUNK_BYTES;
    const uint32_t stage_bytes = p_region + (uint32_t)p.q_chunks * WG_CHUNK_BYTES;
    const uint32_t tx_bytes = (uint32_t)(p_chunks + p.q_chunks) * WG_CHUNK_BYTES;
    const int sub_steps = p.fuse ? 1 : 3;            // pipeline stages per pixel tile

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmZ) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmX) : "memory");
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < p.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        mbar_init(&done_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"((uint32_t)p.tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, tmem_slot, 0);

    if (warp == 0) {
        // ===== TMA producer =====
        int stage = 0; uint32_t phase = 0;
        for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
            const int tw = tile % p.tiles_w, th = (tile / p.tiles_w) % p.tiles_h, n = tile / (p.tiles_w * p.tiles_h);
            const int ow0 = tw * WG_TILE, oh0 = th * WG_TILE;
            const int ix0 = ow0 * p.stride - 1, iy = oh0 * p.stride + frow - 1;
            for (int ss = 0; ss < sub_steps; ++ss) {
                mbar_wait(&empty_bar[stage], phase ^ 1u);
                if (elect_one()) {
                    mbar_arrive_expect_tx(&full_bar[stage], tx_bytes);
                    const uint32_t pb = smem_base + (uint32_t)stage * stage_bytes, qb = pb + p_region;
                    // dz chunks (unshifted operand)
                    const uint32_t zb = p.swap ? qb : pb;
                    const int zc0 = p.swap ? 0 : mt * 4, zn = p.swap ? cout_chunks : p_chunks;
                    for (int c = 0; c < zn; ++c)
                        tma_load_4d(zb + c * WG_CHUNK_BYTES, &tmZ, &full_bar[stage], (zc0 + c) * KCH, ow0, oh0, n);
                    // x chunks (tap-shifted operand): fused -> slots [s][c] for s = 0..2, else slots [c] for s = ss
                    const uint32_t xb = p.swap ? pb : qb;
                    for (int s = (p.fuse ? 0 : ss); s < (p.fuse ? 3 : ss + 1); ++s)
                        for (int c = 0; c < cin_chunks; ++c)
                            tma_load_4d(xb + (uint32_t)((p.fuse ? s * cin_chunks : 0) + c) * WG_CHUNK_BYTES, &tmX, &full_bar[stage],
                                        c * KCH, ix0 + s, iy, n);
                }
                __syncwarp();
                if (++stage == p.stages) { stage = 0; phase ^= 1u; }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: D=f32, A=B=tf32, both MN-major, N = n_mma, M = 128 =====
        const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) |
                               ((uint32_t)(p.n_mma >> 3) << 17) | ((128u >> 4) << 24);
        const uint64_t desc_hi = umma_desc(0, WG_CHUNK_BYTES, 512, 1);
        int stage = 0; uint32_t phase = 0; uint32_t first = 1;
        for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
            for (int ss = 0; ss < sub_steps; ++ss) {
                mbar_wait(&full_bar[stage], phase);
                tc_fence_after();
                const uint32_t pb = smem_base + (uint32_t)stage * stage_bytes, qb = pb + p_region;
                const uint32_t d_tmem = tmem_base + (uint32_t)(ss * p.n_mma);
#pragma unroll
                for (int k8 = 0; k8 < WG_TILE * WG_TILE / 8; ++k8) {
                    tc_mma_tf32_elect(d_tmem, desc_hi | (uint64_t)(((pb + k8 * 1024) & 0x3FFFFu) >> 4),
                                      desc_hi | (uint64_t)(((qb + k8 * 1024) & 0x3FFFFu) >> 4), idesc,
                                      (uint32_t)(!first || k8 != 0));
                }
                tc_commit_elect(&empty_bar[stage]);
                if (++stage == p.stages) { stage = 0; phase ^= 1u; }
            }
            first = 0;
        }
        tc_commit_elect(&done_bar);
    } else if (warp >= 4) {
        // ===== epilogue: TMEM -> registers -> red.global.add into the packed gradient (ORDERED: stores into the slot) =====
        const int q = warp & 3;
        const int m = q * 32 + lane;
        float* const dw = ORDERED ? p.dw + (long)blockIdx.x * 9 * p.Cout * p.Cin : p.dw;
        mbar_wait(&done_bar, 0);
        tc_fence_after();
        for (int a = 0; a < p.accs; ++a) {
            const uint32_t t_row = tmem_base + (uint32_t)(a * p.n_mma) + ((uint32_t)(q * 32) << 16);
            for (int c0 = 0; c0 < p.n_mma; c0 += 32) {
                float v[32];
                tmem_ld32(t_row + c0, v);
                if (!p.swap) {
                    // row = output channel, columns = (tap s, input channel): 32 consecutive ci of one tap
                    const int co = mt * 128 + m;
                    const int s = p.fuse ? c0 / p.Cin : a, ci0 = p.fuse ? c0 % p.Cin : c0;
                    if (co < p.Cout) {
                        const float sc = p.oscale ? p.oscale[co] : 1.f;
                        float* dst = dw + ((long)(frow * 3 + s) * p.Cout + co) * p.Cin + ci0;
#pragma unroll
                        for (int j = 0; j < 32; j += 4) {
                            if (ORDERED)
                                *reinterpret_cast<float4*>(dst + j) = make_float4(v[j] * sc, v[j + 1] * sc, v[j + 2] * sc, v[j + 3] * sc);
                            else
                                asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + j), "f"(v[j] * sc),
                                             "f"(v[j + 1] * sc), "f"(v[j + 2] * sc), "f"(v[j + 3] * sc) : "memory");
                        }
                    }
                } else {
                    // row = (tap s, input channel), columns = output channels: lanes are consecutive ci -> coalesced reds
                    const int s = p.fuse ? m / p.Cin : a, ci = p.fuse ? m % p.Cin : m;
                    if (ci < p.Cin && s < 3 && m < (p.fuse ? 3 * p.Cin : p.Cin)) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const int co = c0 + j;
                            const float sc = p.oscale ? __ldg(p.oscale + co) : 1.f;
                            float* dst = dw + ((long)(frow * 3 + s) * p.Cout + co) * p.Cin + ci;
                            if (ORDERED) *dst = v[j] * sc;
                            else atomicAdd(dst, v[j] * sc);
                        }
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols) : "memory");
    }
}

// slots != NULL: only the plan - *slots = the launch's CTA columns gx (the workspace slots of the ordered form), no launch
int conv_wgrad2_tc_launch(const sci_wgrad_desc* d, void* stream, int* slots = nullptr) {
    Wgrad2Params p;
    p.oscale = d->oscale; p.dw = d->dw;
    p.N = d->N; p.stride = d->stride; p.Cin = d->Cin; p.Cout = d->Cout;
    p.Ho = (d->H - 1) / d->stride + 1; p.Wo = (d->W - 1) / d->stride + 1;
    p.tiles_w = (p.Wo + WG_TILE - 1) / WG_TILE; p.tiles_h = (p.Ho + WG_TILE - 1) / WG_TILE;
    p.num_tiles = p.tiles_w * p.tiles_h * p.N;
    const int cin_chunks = p.Cin / KCH, cout_chunks = p.Cout / KCH;
    // orientation: put the wider channel dimension on the (128-row padded) M side
    p.swap = (p.Cout < p.Cin || (p.Cin == 32 && p.Cout == 32)) ? 1 : 0;
    if (p.swap) {
        p.fuse = (3 * p.Cin <= 128) ? 1 : 0;                   // taps stacked along M
        p.p_chunks = p.fuse ? 3 * cin_chunks : cin_chunks;
        p.q_chunks = cout_chunks;
        p.n_mma = p.Cout;
        p.accs = p.fuse ? 1 : 3;
        p.m_tiles = 1;
    } else {
        p.fuse = (3 * p.Cin <= 256) ? 1 : 0;                   // taps side by side along N
        p.p_chunks = 0;                                        // per-CTA (depends on the M tile)
        p.q_chunks = p.fuse ? 3 * cin_chunks : cin_chunks;
        p.n_mma = p.fuse ? 3 * p.Cin : p.Cin;
        p.accs = p.fuse ? 1 : 3;
        p.m_tiles = (p.Cout + 127) / 128;
    }
    if (p.swap && (p.Cin > 128 || p.Cout > 256)) return sci_fail(SCI_EUNSUPPORTED, "wgrad tc v2: shape");
    p.tmem_cols = next_pow2_cols(p.accs * p.n_mma);
    if (p.tmem_cols > 512) return sci_fail(SCI_EUNSUPPORTED, "wgrad tc v2: accumulators exceed TMEM");
    const size_t stage_bytes = (size_t)4 * WG_CHUNK_BYTES + (size_t)p.q_chunks * WG_CHUNK_BYTES;
    p.stages = (int)min((size_t)4, (size_t)(214 * 1024) / stage_bytes);
    if (p.stages < 2) return sci_fail(SCI_EUNSUPPORTED, "wgrad tc v2: pipeline does not fit");
    const int groups = 3 * p.m_tiles;
    const int gx = max(1, min(p.num_tiles, SCI_NUM_SMS / groups));
    if (slots) { *slots = gx; return SCI_OK; }
    CUtensorMap tmZ, tmX;
    int rc = make_act_map(&tmZ, d->dz, d->N, p.Ho, p.Wo, d->Cout, 1, WG_TILE, WG_TILE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B);
    if (rc) return rc;
    rc = make_act_map(&tmX, d->x, d->N, d->H, d->W, d->Cin, d->stride, WG_TILE, WG_TILE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B);
    if (rc) return rc;
    const size_t smem = p.stages * stage_bytes + 1024;
    if (env_int("SCI_CONV_VERBOSE", 0))
        fprintf(stderr, "wgrad v2 plan: %dx%d Cin %d Cout %d stride %d | swap %d fuse %d m_tiles %d accs %d stages %d grid %d groups %d tiles %d\n",
                d->H, d->W, d->Cin, d->Cout, d->stride, p.swap, p.fuse, p.m_tiles, p.accs, p.stages, gx, groups, p.num_tiles);
    if (d->workspace) {
        p.dw = static_cast<float*>(d->workspace);
        rc = launch(conv_wgrad2_tc_kernel<true>, dim3(gx, groups), TC_THREADS, smem, stream, false, "conv tc wgrad v2", tmZ, tmX, p);
        return rc ? rc : sci_ordered_slot_sum(p.dw, gx, 9L * p.Cout * p.Cin, 9L * p.Cout * p.Cin, d->dw, nullptr, stream);
    }
    return launch(conv_wgrad2_tc_kernel<false>, dim3(gx, groups), TC_THREADS, smem, stream, false, "conv tc wgrad v2", tmZ, tmX, p);
}

// ---------------------------------------------------------------------------------------------------
// weight-gradient kernel, version 3 ("rs-stack"): all nine taps in ONE CTA, one pass over the data
//   dW[r,s][co][ci] = sum_p dz[p][co] * x[p + (r-1) rows + (s-1) cols][ci]
//   Version 2 ran one filter row per CTA group: dz and x were read three times, and with 32-channel layers only a quarter
//   of the MMA rows did useful work (full-resolution layers: 0.47-0.86 ms each, 60 % of the weight-gradient time).
//   Here the operand with FEWER channels (P) goes on the M side as the stack of its three ROW-shifted views - one
//   {32 ch, 8 px, 10 rows} box per 32-channel chunk; a row shift is 1024 bytes, the swizzle period, so the views are plain
//   descriptor offsets and the stack has a uniform leading-dimension stride of 1024 bytes - and the other operand (Q) on
//   the N side as the stack of its three COLUMN-shifted 8x8 boxes.  One MMA per 8 pixels then yields the 3x3 block of
//   taps for 32 P-channels x all Q-channels:  D[(r, p-ch)][(s, q-ch)].
//     case A (P = dz, Q = x):  sum over q of dz[q - (r-1) rows] * x[q + (s-1) cols]   -> P view r starts at box row 2-r
//     case B (P = x, Q = dz):  sum over q of x[q + (r-1) rows] * dz[q - (s-1) cols]   -> P view r starts at box row r
//   TMA zero fill supplies both the conv padding (x) and the out-of-image output pixels (dz).
// ---------------------------------------------------------------------------------------------------
constexpr int WG3_P_BYTES = 10 * 1024;           // P chunk box: 10 rows x 8 px x 128 B
struct Wgrad3Params {
    const float* oscale; float* dw;
    int N, H, W, Cin, Cout;
    int tiles_w, tiles_h, num_tiles;
    int p_is_dz, p_chunks, q_chunks, q_slots, n_tot, tmem_cols, stages;
};

template <bool ORDERED>
__global__ void __launch_bounds__(TC_THREADS, 1)
conv_wgrad3_tc_kernel(const __grid_constant__ CUtensorMap tmP, const __grid_constant__ CUtensorMap tmQ, const Wgrad3Params p) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[4], empty_bar[4], done_bar;
    __shared__ uint32_t tmem_slot;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t p_bytes = (uint32_t)p.p_chunks * WG3_P_BYTES, q_bytes = (uint32_t)p.q_slots * WG_CHUNK_BYTES;
    const uint32_t stage_bytes = p_bytes + q_bytes;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmP) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmQ) : "memory");
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < p.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        mbar_init(&done_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"((uint32_t)p.tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, tmem_slot, 0);

    if (warp == 0) {
        // ===== TMA producer =====
        int stage = 0; uint32_t phase = 0;
        for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
            const int tw = tile % p.tiles_w, th = (tile / p.tiles_w) % p.tiles_h, n = tile / (p.tiles_w * p.tiles_h);
            const int ow0 = tw * WG_TILE, oh0 = th * WG_TILE;
            mbar_wait(&empty_bar[stage], phase ^ 1u);
            if (elect_one()) {
                mbar_arrive_expect_tx(&full_bar[stage], stage_bytes);
                const uint32_t pb = smem_base + (uint32_t)stage * stage_bytes, qb = pb + p_bytes;
                for (int c = 0; c < p.p_chunks; ++c)
                    tma_load_4d(pb + (uint32_t)c * WG3_P_BYTES, &tmP, &full_bar[stage], c * KCH, ow0, oh0 - 1, n);
                for (int s = 0; s < 3; ++s)
                    for (int c = 0; c < p.q_chunks; ++c)
                        tma_load_4d(qb + (uint32_t)(s * p.q_chunks + c) * WG_CHUNK_BYTES, &tmQ, &full_bar[stage], c * KCH,
                                    ow0 + (p.p_is_dz ? s - 1 : 1 - s), oh0, n);
            }
            __syncwarp();
            if (++stage == p.stages) { stage = 0; phase ^= 1u; }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: both operands MN-major (SWIZZLE_128B_BASE32B), M = 128 (rows 96..127 unused), K = 8 pixels =====
        const uint32_t idesc0 = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | ((128u >> 4) << 24);
        const uint64_t pdesc_hi = umma_desc(0, 1024, 512, 1);              // stack of row-shifted views: stride 1024 B
        const uint64_t qdesc_hi = umma_desc(0, WG_CHUNK_BYTES, 512, 1);    // stack of boxes: stride 8192 B
        int stage = 0; uint32_t phase = 0; uint32_t first = 1;
        for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
            mbar_wait(&full_bar[stage], phase);
            tc_fence_after();
            const uint32_t pb = smem_base + (uint32_t)stage * stage_bytes, qb = pb + p_bytes;
            for (int c = 0; c < p.p_chunks; ++c) {
                for (int g0 = 0; g0 < p.q_slots; g0 += 8) {                 // N groups of <= 8 slots (256 columns)
                    const int ns = min(8, p.q_slots - g0);
                    const uint32_t idesc = idesc0 | ((uint32_t)((ns * 32) >> 3) << 17);
                    const uint32_t d_tmem = tmem_base + (uint32_t)(c * p.n_tot + g0 * 32);
                    const uint32_t a0 = pb + (uint32_t)c * WG3_P_BYTES, b0 = qb + (uint32_t)g0 * WG_CHUNK_BYTES;
#pragma unroll
                    for (int k8 = 0; k8 < WG_TILE; ++k8) {
                        tc_mma_tf32_elect(d_tmem, pdesc_hi | (uint64_t)(((a0 + k8 * 1024) & 0x3FFFFu) >> 4),
                                          qdesc_hi | (uint64_t)(((b0 + k8 * 1024) & 0x3FFFFu) >> 4), idesc,
                                          (uint32_t)(!first || k8 != 0));
                    }
                }
            }
            tc_commit_elect(&empty_bar[stage]);
            if (++stage == p.stages) { stage = 0; phase ^= 1u; }
            first = 0;
        }
        tc_commit_elect(&done_bar);
    } else if (warp >= 4) {
        // ===== epilogue: TMEM -> registers -> red.global.add into the packed gradient dw[tap][co][ci] (ORDERED: plain stores
        // into slot blockIdx.x of the [gx][9][Cout][Cin] workspace at p.dw; each CTA covers the whole slot) =====
        const int i = warp & 3;                        // stacked view index: TMEM lanes 32 i .. 32 i + 31
        float* const dw = ORDERED ? p.dw + (long)blockIdx.x * 9 * p.Cout * p.Cin : p.dw;
        if (i < 3 && blockIdx.x < p.num_tiles) {
            mbar_wait(&done_bar, 0);
            tc_fence_after();
            const int r = p.p_is_dz ? 2 - i : i;
            for (int c = 0; c < p.p_chunks; ++c) {
                const int pch = c * 32 + lane;
                const uint32_t t_row = tmem_base + (uint32_t)(c * p.n_tot) + ((uint32_t)(i * 32) << 16);
                for (int slot = 0; slot < p.q_slots; ++slot) {
                    float v[32];
                    tmem_ld32(t_row + slot * 32, v);
                    const int s = slot / p.q_chunks, q0 = (slot % p.q_chunks) * 32;
                    const int tap = r * 3 + s;
                    if (p.p_is_dz) {                   // row = output channel, 32 consecutive input channels
                        const float sc = p.oscale ? p.oscale[pch] : 1.f;
                        float* dst = dw + ((long)tap * p.Cout + pch) * p.Cin + q0;
#pragma unroll
                        for (int j = 0; j < 32; j += 4) {
                            if (ORDERED)
                                *reinterpret_cast<float4*>(dst + j) = make_float4(v[j] * sc, v[j + 1] * sc, v[j + 2] * sc, v[j + 3] * sc);
                            else
                                asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + j), "f"(v[j] * sc),
                                             "f"(v[j + 1] * sc), "f"(v[j + 2] * sc), "f"(v[j + 3] * sc) : "memory");
                        }
                    } else {                           // row = input channel (lanes consecutive -> coalesced), 32 output channels
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const int co = q0 + j;
                            const float sc = p.oscale ? __ldg(p.oscale + co) : 1.f;
                            float* dst = dw + ((long)tap * p.Cout + co) * p.Cin + pch;
                            if (ORDERED) *dst = v[j] * sc;
                            else atomicAdd(dst, v[j] * sc);
                        }
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols) : "memory");
    }
}

bool wgrad3_eligible(const sci_wgrad_desc* d) {
    const int cp = min(d->Cin, d->Cout), cq = max(d->Cin, d->Cout);
    return d->stride == 1 && (cp == 32 || cp == 64) && cq <= 96 && (cp / 32) * 3 * cq <= 512 && env_int("SCI_WGRAD_V3", 1) != 0;
}

// slots: as conv_wgrad2_tc_launch
int conv_wgrad3_tc_launch(const sci_wgrad_desc* d, void* stream, int* slots = nullptr) {
    Wgrad3Params p;
    p.oscale = d->oscale; p.dw = d->dw;
    p.N = d->N; p.H = d->H; p.W = d->W; p.Cin = d->Cin; p.Cout = d->Cout;
    p.tiles_w = (p.W + WG_TILE - 1) / WG_TILE; p.tiles_h = (p.H + WG_TILE - 1) / WG_TILE;
    p.num_tiles = p.tiles_w * p.tiles_h * p.N;
    p.p_is_dz = d->Cout <= d->Cin ? 1 : 0;
    const int cp = p.p_is_dz ? d->Cout : d->Cin, cq = p.p_is_dz ? d->Cin : d->Cout;
    p.p_chunks = cp / KCH; p.q_chunks = cq / KCH; p.q_slots = 3 * p.q_chunks; p.n_tot = 3 * cq;
    p.tmem_cols = next_pow2_cols(p.p_chunks * p.n_tot);
    const size_t stage_bytes = (size_t)p.p_chunks * WG3_P_BYTES + (size_t)p.q_slots * WG_CHUNK_BYTES;
    // the 4th (unused) stacked view of the last k-step reads up to 1 KB past the P box: keep a guard after the ring
    p.stages = (int)min((size_t)4, (size_t)(212 * 1024) / stage_bytes);
    if (p.stages < 2) return sci_fail(SCI_EUNSUPPORTED, "wgrad tc v3: pipeline does not fit");
    const int gx = max(1, min(p.num_tiles, SCI_NUM_SMS));
    if (slots) { *slots = gx; return SCI_OK; }
    CUtensorMap tmP, tmQ;
    const float* P = p.p_is_dz ? d->dz : d->x;
    const float* Q = p.p_is_dz ? d->x : d->dz;
    int rc = make_act_map(&tmP, P, d->N, d->H, d->W, cp, 1, WG_TILE, 10, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B);
    if (rc) return rc;
    rc = make_act_map(&tmQ, Q, d->N, d->H, d->W, cq, 1, WG_TILE, WG_TILE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B);
    if (rc) return rc;
    const size_t smem = p.stages * stage_bytes + 2048 + 1024;
    if (env_int("SCI_CONV_VERBOSE", 0))
        fprintf(stderr, "wgrad v3 plan: %dx%d Cin %d Cout %d stride 1 | p_is_dz %d cp %d cq %d stages %d grid %d tiles %d\n", d->H, d->W,
                d->Cin, d->Cout, p.p_is_dz, cp, cq, p.stages, gx, p.num_tiles);
    if (d->workspace) {
        p.dw = static_cast<float*>(d->workspace);
        rc = launch(conv_wgrad3_tc_kernel<true>, dim3(gx), TC_THREADS, smem, stream, false, "conv tc wgrad v3", tmP, tmQ, p);
        return rc ? rc : sci_ordered_slot_sum(p.dw, gx, 9L * p.Cout * p.Cin, 9L * p.Cout * p.Cin, d->dw, nullptr, stream);
    }
    return launch(conv_wgrad3_tc_kernel<false>, dim3(gx), TC_THREADS, smem, stream, false, "conv tc wgrad v3", tmP, tmQ, p);
}

int check_conv_desc(const sci_conv_desc* d) {
    SCI_REQUIRE(d && d->x && d->w && (d->y || d->planar_out), "conv: null pointer");
    SCI_REQUIRE(!d->planar_out || (d->stride == 1 && !d->w_split && !d->emit_lo), "conv: planar output options");
    SCI_REQUIRE(d->planar_planes == 0 || d->planar_planes == 1 || d->planar_planes == 3, "conv: planar_planes 0, 1 or 3");
    SCI_REQUIRE(d->N > 0 && d->H > 0 && d->W > 0 && d->Cin > 0 && d->Cout > 0, "conv: shape");
    SCI_REQUIRE(d->Cin % 8 == 0 && d->Cout % 4 == 0, "conv: Cin % 8, Cout % 4");
    SCI_REQUIRE(!d->half_io || ((d->Cin % 64 == 0 || d->Cin == 32) && d->Cout % 32 == 0 && !d->emit_lo), "conv fp16: Cin % 64 (or 32), Cout % 32, no emit_lo");
    SCI_REQUIRE(!(d->half_io && d->w_split) || (d->stride == 1 && d->Cin % 64 == 0), "conv fp16 split form (w_split): stride 1, Cin = 64 per group of 32 channels");
    SCI_REQUIRE(d->stride == 1 || d->stride == 2, "conv: stride");
    SCI_REQUIRE(!d->pixel_shuffle || d->stride == 1, "conv: pixel_shuffle with stride 2");
    return SCI_OK;
}

}  // namespace

extern "C" int sci_conv_tc_available(void) { return 1; }

extern "C" size_t sci_conv3x3_fwd_workspace_bytes(const sci_conv_desc* d, int impl) {
    if (!d || impl != SCI_CONV_TC || !d->mask_y || !d->col_s1 || check_conv_desc(d) || !fwd2_eligible(d)) return 0;
    const int halves = d->Cout <= 128 ? 1 : 2;
    int grid = 0;
    if (conv_fwd2_tc_launch(d, nullptr, 0, halves == 1 ? d->Cout : 128, nullptr, &grid, true)) return 0;
    const int ncol = d->pixel_shuffle ? d->Cout / 4 : d->Cout;
    return (size_t)halves * grid * 2 * ncol * sizeof(float);
}

extern "C" int sci_conv3x3_fwd(const sci_conv_desc* d, int impl, void* stream) {
    int rc = check_conv_desc(d);
    if (rc) return rc;
    size_t need = 0;
    if (d->workspace || d->workspace_bytes) {
        need = sci_conv3x3_fwd_workspace_bytes(d, impl);
        SCI_REQUIRE(d->workspace && d->workspace_bytes >= need, "conv ordered column sums: workspace missing or too small");
        SCI_REQUIRE(((uintptr_t)d->workspace & 15) == 0, "conv ordered column sums: workspace must be 16-byte aligned");
    }
    if (impl == SCI_CONV_REF) {
        SCI_REQUIRE(!d->w_split && !d->emit_lo && !d->planar_out && !d->half_io, "conv ref: w_split / emit_lo / planar_out / half_io are tensor-core options");
        return sci_conv3x3_ref_launch(d, stream);
    }
    if (impl == SCI_CONV_TC) {
        if (!fwd2_eligible(d)) return conv_fwd_tc_launch(d, stream);
        float* ord = need ? static_cast<float*>(d->workspace) : nullptr;
        const int ncol = d->pixel_shuffle ? d->Cout / 4 : d->Cout;       // stored channels: the column sums' width
        int grid = 0;
        if (d->Cout <= 128) {
            rc = conv_fwd2_tc_launch(d, stream, 0, d->Cout, ord, &grid);
        } else {
            // 256 columns: two passes of 128 (PixelShuffle layers: the two output-row parities); the activation rows are
            // fetched twice, the tensor-core work is unchanged.  Ordered sums: the second pass has the slots after the first's
            rc = conv_fwd2_tc_launch(d, stream, 0, 128, ord, &grid);
            if (!rc) rc = conv_fwd2_tc_launch(d, stream, 128, 128, ord ? ord + (size_t)grid * 2 * ncol : nullptr);
        }
        if (rc || !ord) return rc;
        return sci_ordered_slot_sum(ord, (d->Cout <= 128 ? 1 : 2) * grid, 2L * ncol, ncol, d->col_s1, d->col_s2, stream);
    }
    return sci_fail(SCI_EINVAL, "conv: unknown impl");
}

extern "C" int sci_conv3x3_dgrad(const sci_conv_desc* d, int impl, void* stream) {
    return sci_conv3x3_fwd(d, impl, stream);
}

static int check_wgrad_desc(const sci_wgrad_desc* d, int impl) {
    SCI_REQUIRE(d && d->x && d->dz && d->dw, "wgrad: null pointer");
    SCI_REQUIRE(d->N > 0 && d->H > 0 && d->W > 0 && d->Cin > 0 && d->Cout > 0 && (d->stride == 1 || d->stride == 2),
                "wgrad: shape");
    SCI_REQUIRE(d->Cin % 4 == 0 && d->Cout % 4 == 0, "wgrad: channels % 4");
    if (impl == SCI_CONV_TC && (d->Cin % 32 != 0 || d->Cout % 32 != 0 || d->Cin > 128 || d->Cout > 256))
        return sci_fail(SCI_EUNSUPPORTED, "wgrad tc: needs Cin % 32 == 0 (<= 128), Cout % 32 == 0 (<= 256)");
    if (impl != SCI_CONV_TC && impl != SCI_CONV_REF) return sci_fail(SCI_EINVAL, "wgrad: unknown impl");
    return SCI_OK;
}

// CTA columns of the weight-gradient launch = slots of its ordered form (0: the descriptor is rejected)
static int wgrad_slots(const sci_wgrad_desc* d, int impl) {
    if (check_wgrad_desc(d, impl)) return 0;
    if (impl == SCI_CONV_REF) return sci_wgrad_ref_slots(d);
    int slots = 0;
    const int rc = wgrad3_eligible(d) ? conv_wgrad3_tc_launch(d, nullptr, &slots) : conv_wgrad2_tc_launch(d, nullptr, &slots);
    return rc ? 0 : slots;
}

extern "C" size_t sci_conv3x3_wgrad_workspace_bytes(const sci_wgrad_desc* d, int impl) {
    const int slots = wgrad_slots(d, impl);
    return slots ? (size_t)slots * 9 * (size_t)d->Cout * (size_t)d->Cin * sizeof(float) : 0;
}

extern "C" int sci_conv3x3_wgrad(const sci_wgrad_desc* d, int impl, void* stream) {
    int rc = check_wgrad_desc(d, impl);
    if (rc) return rc;
    if (d->workspace || d->workspace_bytes) {
        const size_t need = sci_conv3x3_wgrad_workspace_bytes(d, impl);
        SCI_REQUIRE(d->workspace && d->workspace_bytes >= need, "wgrad ordered: workspace missing or too small");
        SCI_REQUIRE(((uintptr_t)d->workspace & 15) == 0, "wgrad ordered: workspace must be 16-byte aligned");
    }
    if (impl == SCI_CONV_REF) return sci_wgrad_ref_launch(d, stream);
    if (wgrad3_eligible(d)) return conv_wgrad3_tc_launch(d, stream);
    return conv_wgrad2_tc_launch(d, stream);
}
