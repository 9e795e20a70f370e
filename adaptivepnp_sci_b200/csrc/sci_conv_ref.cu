// fp32 FFMA implicit-GEMM 3x3 convolution (forward / data-gradient / weight-gradient).
//
// This is the ON-DEVICE NUMERICS REFERENCE for the tensor-core kernels in sci_conv_tc.cu
// (impl = SCI_CONV_REF): same descriptors, same layouts, plain fp32 arithmetic.  The
// product path (impl = SCI_CONV_TC) never routes through it; tests use it to separate
// "TF32 rounding" from "kernel bug", and the engine can be switched to it as a whole for
// fp32-exact fine-tune parity runs.
#include "sci_common.cuh"

namespace {

constexpr int RT = 8;     // 8x8 output pixels per block
constexpr int RCO = 64;   // output columns per block
constexpr int RCI = 8;    // input-channel chunk
constexpr int RPMAX = (RT - 1) * 2 + 3;   // 17: input patch edge for stride 2

__device__ __forceinline__ float round_tf32_rna(float v) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
    return __uint_as_float(r);
}

__global__ void __launch_bounds__(256) conv3x3_ref_kernel(sci_conv_desc d) {
    __shared__ float sA[RPMAX][RPMAX][RCI];
    __shared__ float sB[9][RCI][RCO];
    const int Ho = (d.H - 1) / d.stride + 1, Wo = (d.W - 1) / d.stride + 1;
    const int tiles_w = (Wo + RT - 1) / RT;
    const int th0 = (blockIdx.x / tiles_w) * RT, tw0 = (blockIdx.x % tiles_w) * RT;
    const int co0 = blockIdx.y * RCO, n = blockIdx.z;
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
    const int P = (RT - 1) * d.stride + 3;
    const int ih0 = th0 * d.stride - 1, iw0 = tw0 * d.stride - 1;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    int ph[4], pw[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) { const int p = ty * 4 + i; ph[i] = (p / RT) * d.stride; pw[i] = (p % RT) * d.stride; }

    for (int ci0 = 0; ci0 < d.Cin; ci0 += RCI) {
        for (int i = tid; i < P * P * RCI; i += 256) {
            const int c = i % RCI, pc = (i / RCI) % P, pr = i / (RCI * P);
            const int ih = ih0 + pr, iw = iw0 + pc;
            float v = 0.f;
            if (ih >= 0 && ih < d.H && iw >= 0 && iw < d.W)
                v = d.x[(((long)n * d.H + ih) * d.W + iw) * d.Cin + ci0 + c];
            sA[pr][pc][c] = v;
        }
        for (int i = tid; i < 9 * RCO * RCI; i += 256) {
            const int c = i % RCI, co = (i / RCI) % RCO, tap = i / (RCI * RCO);
            float v = 0.f;
            if (co0 + co < d.Cout) v = d.w[((long)tap * d.Cout + co0 + co) * d.Cin + ci0 + c];
            sB[tap][c][co] = v;
        }
        __syncthreads();
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) {
            const int r = tap / 3, q = tap % 3;
#pragma unroll
            for (int c = 0; c < RCI; ++c) {
                const float4 bv = *reinterpret_cast<const float4*>(&sB[tap][c][tx * 4]);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float a = sA[ph[i] + r][pw[i] + q][c];
                    acc[i][0] += a * bv.x; acc[i][1] += a * bv.y; acc[i][2] += a * bv.z; acc[i][3] += a * bv.w;
                }
            }
        }
        __syncthreads();
    }
    const int Cq = d.Cout >> 2;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int p = ty * 4 + i, ho = th0 + p / RT, wo = tw0 + p % RT;
        if (ho >= Ho || wo >= Wo) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int co = co0 + tx * 4 + j;
            if (co >= d.Cout) continue;
            float v = acc[i][j];
            if (d.scale) v = v * d.scale[co];
            if (d.shift) v = v + d.shift[co];
            if (d.relu) v = fmaxf(v, 0.f);
            long o;
            if (d.pixel_shuffle) {
                const int qq = co / Cq, c = co % Cq;
                o = (((long)n * 2 * Ho + 2 * ho + (qq >> 1)) * 2 * Wo + 2 * wo + (qq & 1)) * Cq + c;
            } else {
                o = (((long)n * Ho + ho) * Wo + wo) * d.Cout + co;
            }
            if (d.residual) v = v + d.residual[o];
            if (d.round_tf32) v = round_tf32_rna(v);
            d.y[o] = v;
        }
    }
}

// Weight gradient: one block = one tap x (64 co x 64 ci) tile x one chunk of output pixels.
// ORDERED: d.dw points at slot 0 of a [chunks][9][Cout][Cin] workspace; pixel chunk b stores its partial into slot b
// (sci_ordered_slot_sum then adds the slots in order) instead of adding it into dw with atomics.
constexpr int WG_PIX = 16;
template <bool ORDERED>
__global__ void __launch_bounds__(256) wgrad_ref_kernel(sci_wgrad_desc d, int pix_per_block) {
    __shared__ float sZ[WG_PIX][64];
    __shared__ float sX[WG_PIX][64];
    const int Ho = (d.H - 1) / d.stride + 1, Wo = (d.W - 1) / d.stride + 1;
    const long npix = (long)d.N * Ho * Wo;
    const int tap = blockIdx.y, r = tap / 3, q = tap % 3;
    const int ci_tiles = (d.Cin + 63) / 64;
    const int co0 = (blockIdx.z / ci_tiles) * 64, ci0 = (blockIdx.z % ci_tiles) * 64;
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    const long p_begin = (long)blockIdx.x * pix_per_block;
    const long p_end = min(npix, p_begin + pix_per_block);
    for (long p0 = p_begin; p0 < p_end; p0 += WG_PIX) {
        for (int i = tid; i < WG_PIX * 64; i += 256) {
            const int c = i & 63, pp = i >> 6;
            const long p = p0 + pp;
            float zv = 0.f, xv = 0.f;
            if (p < p_end) {
                const int wo = (int)(p % Wo), ho = (int)((p / Wo) % Ho), n = (int)(p / ((long)Wo * Ho));
                if (co0 + c < d.Cout) zv = d.dz[p * d.Cout + co0 + c];
                const int ih = ho * d.stride + r - 1, iw = wo * d.stride + q - 1;
                if (ci0 + c < d.Cin && ih >= 0 && ih < d.H && iw >= 0 && iw < d.W)
                    xv = d.x[(((long)n * d.H + ih) * d.W + iw) * d.Cin + ci0 + c];
            }
            sZ[pp][c] = zv; sX[pp][c] = xv;
        }
        __syncthreads();
#pragma unroll
        for (int pp = 0; pp < WG_PIX; ++pp) {
            const float4 zv = *reinterpret_cast<const float4*>(&sZ[pp][ty * 4]);
            const float4 xv = *reinterpret_cast<const float4*>(&sX[pp][tx * 4]);
            const float z[4] = {zv.x, zv.y, zv.z, zv.w}, xx[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] += z[i] * xx[j];
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int co = co0 + ty * 4 + i;
        if (co >= d.Cout) continue;
        const float s = d.oscale ? d.oscale[co] : 1.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int ci = ci0 + tx * 4 + j;
            if (ci >= d.Cin) continue;
            if (ORDERED) d.dw[((long)blockIdx.x * 9 + tap) * d.Cout * d.Cin + (long)co * d.Cin + ci] = s * acc[i][j];
            else atomicAdd(&d.dw[((long)tap * d.Cout + co) * d.Cin + ci], s * acc[i][j]);
        }
    }
}

}  // namespace

int sci_conv3x3_ref_launch(const sci_conv_desc* d, void* stream) {
    const int Ho = (d->H - 1) / d->stride + 1, Wo = (d->W - 1) / d->stride + 1;
    const dim3 grid(((Wo + RT - 1) / RT) * ((Ho + RT - 1) / RT), (d->Cout + RCO - 1) / RCO, d->N);
    if (grid.z > 65535) return sci_fail(SCI_EUNSUPPORTED, "conv ref: batch too large");
    conv3x3_ref_kernel<<<grid, 256, 0, sci_stream(stream)>>>(*d);
    SCI_CHECK_LAUNCH("conv3x3 ref");
    return SCI_OK;
}

// pixel chunks of the weight-gradient launch (its grid.x) and the pixels per chunk
static int wgrad_ref_chunks(const sci_wgrad_desc* d, int* ppb_out) {
    const int Ho = (d->H - 1) / d->stride + 1, Wo = (d->W - 1) / d->stride + 1;
    const long npix = (long)d->N * Ho * Wo;
    int chunks = (int)min((long)SCI_NUM_SMS * 2, (npix + 255) / 256);
    const int ppb = (int)((npix + chunks - 1) / chunks);
    const int ppb_al = ((ppb + WG_PIX - 1) / WG_PIX) * WG_PIX;
    if (ppb_out) *ppb_out = ppb_al;
    return (int)((npix + ppb_al - 1) / ppb_al);
}

int sci_wgrad_ref_slots(const sci_wgrad_desc* d) { return wgrad_ref_chunks(d, nullptr); }

int sci_wgrad_ref_launch(const sci_wgrad_desc* d, void* stream) {
    int ppb_al = 0;
    const int chunks = wgrad_ref_chunks(d, &ppb_al);
    const dim3 grid(chunks, 9, ((d->Cout + 63) / 64) * ((d->Cin + 63) / 64));
    if (d->workspace) {
        sci_wgrad_desc o = *d;
        o.dw = static_cast<float*>(d->workspace);
        wgrad_ref_kernel<true><<<grid, 256, 0, sci_stream(stream)>>>(o, ppb_al);
        SCI_CHECK_LAUNCH("wgrad ref");
        return sci_ordered_slot_sum(o.dw, chunks, 9L * d->Cout * d->Cin, 9L * d->Cout * d->Cin, d->dw, nullptr, stream);
    }
    wgrad_ref_kernel<false><<<grid, 256, 0, sci_stream(stream)>>>(*d, ppb_al);
    SCI_CHECK_LAUNCH("wgrad ref");
    return SCI_OK;
}
