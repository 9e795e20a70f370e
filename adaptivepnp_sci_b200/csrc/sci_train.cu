// Glue kernels of the denoiser engine: weight packing, BatchNorm folding, activation backward,
// network-boundary packers (FFDNet pixel-(un)shuffle + sigma map, FastDVDnet circular frame
// triples + residual output), the fused measurement-consistency loss, and Adam.
// All HBM-bound elementwise / index-remap work; compiled with --fmad=false.
#include <cuda_fp16.h>

#include "sci_common.cuh"

namespace {

__device__ __forceinline__ float rna_tf32(float v) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
    return __uint_as_float(r);
}

// column of the GEMM output that holds PyTorch output channel co.  PixelShuffle layers: the four sub-pixel groups are
// Co_pad/4 columns wide each (the up-sampled tensor's padded channel count), channel co -> group co&3, slot co>>2
__device__ __forceinline__ int out_column(int co, int Co_pad, int ps) {
    return ps ? (co & 3) * (Co_pad >> 2) + (co >> 2) : co;
}

__global__ void pack_weights_kernel(const float* __restrict__ w, float* __restrict__ packed, int Co, int Ci, int groups,
                                    int Co_pad, int Ci_pad, int ps, const float* __restrict__ oscale, int tflip,
                                    int round_tf32, int ci_dup) {
    const long total = (long)9 * Co_pad * Ci_pad;
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    int tap, col, ci;
    if (!tflip) { ci = (int)(idx % Ci_pad); col = (int)((idx / Ci_pad) % Co_pad); tap = (int)(idx / ((long)Ci_pad * Co_pad)); }
    else        { col = (int)(idx % Co_pad); ci = (int)((idx / Co_pad) % Ci_pad); tap = (int)(idx / ((long)Ci_pad * Co_pad)); }
    float v = 0.f;
    if (ci_dup > 0 && ci >= ci_dup && ci < ci_dup + Ci) ci -= ci_dup;     // remainder copy of the input: same weights
    // invert the column permutation: which torch channel lives in this column?
    const int q = Co_pad >> 2;
    const int co = ps ? (col % q) * 4 + col / q : col;
    if ((ps ? (col % q) < (Co >> 2) : col < Co) && ci < Ci) {
        const int cig = Ci / groups, cog = Co / groups, g = co / cog;
        if (ci / cig == g) {
            const int src_tap = tflip ? 8 - tap : tap;
            v = w[((long)co * cig + (ci - g * cig)) * 9 + src_tap];
            if (tflip && oscale) v = v * oscale[col];
        }
    }
    if (round_tf32 == 2) {              // split form: hi in taps 0..8, remainder in taps 9..17
        const float hi = rna_tf32(v);
        packed[idx] = hi;
        packed[idx + total] = rna_tf32(v - hi);
        return;
    }
    if (round_tf32) v = rna_tf32(v);
    packed[idx] = v;
}

// Data gradient of a STRIDE-2 convolution as a sub-pixel convolution at the LOW resolution (no zero-dilated tensor):
//   z[i,j] = sum_{kh,kw} w[kh,kw] x[2i+kh-1, 2j+kw-1]   =>   dx[2i'+a, 2j'+b] = sum over the taps whose parity matches:
//   a = 0: kh = 1 (from dz[i']);   a = 1: kh = 2 (from dz[i']) and kh = 0 (from dz[i'+1]);   same for b / kw.
// Written as a 3x3 correlation over dz with 4*Ci_pad output columns (sub-pixel q = a*2+b, column q*Ci_pad + ci) whose
// result the conv kernels scatter with their PixelShuffle epilogue.  packed[tap][col][co], tap = (dh+1)*3 + (dw+1).
__device__ __forceinline__ int s2t_src_tap(int par, int d) {      // kernel index feeding output parity `par` from offset d
    if (par == 0) return d == 0 ? 1 : -1;
    return d == 0 ? 2 : (d == 1 ? 0 : -1);
}
__global__ void pack_weights_s2t_kernel(const float* __restrict__ w, float* __restrict__ packed, int Co, int Ci, int Co_pad,
                                        int Ci_pad, const float* __restrict__ oscale, int round_tf32) {
    const long total = (long)9 * 4 * Ci_pad * Co_pad;
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int co = (int)(idx % Co_pad);
    const int col = (int)((idx / Co_pad) % (4 * Ci_pad));
    const int tap = (int)(idx / ((long)Co_pad * 4 * Ci_pad));
    const int q = col / Ci_pad, ci = col % Ci_pad;
    const int kh = s2t_src_tap(q >> 1, tap / 3 - 1), kw = s2t_src_tap(q & 1, tap % 3 - 1);
    float v = 0.f;
    if (co < Co && ci < Ci && kh >= 0 && kw >= 0) {
        v = w[((long)co * Ci + ci) * 9 + kh * 3 + kw];
        if (oscale) v = v * oscale[co];
    }
    packed[idx] = round_tf32 ? rna_tf32(v) : v;
}

__global__ void unpack_wgrad_kernel(const float* __restrict__ packed, float* __restrict__ dw, int Co, int Ci, int groups,
                                    int Co_pad, int Ci_pad, int ps, int ci_dup) {
    const int cig = Ci / groups, cog = Co / groups;
    const long total = (long)Co * cig * 9;
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int tap = (int)(idx % 9), cil = (int)((idx / 9) % cig), co = (int)(idx / (9L * cig));
    const int ci = (co / cog) * cig + cil;
    const int col = out_column(co, Co_pad, ps);
    float g = packed[((long)tap * Co_pad + col) * Ci_pad + ci];
    if (ci_dup > 0) g += packed[((long)tap * Co_pad + col) * Ci_pad + ci + ci_dup];
    dw[idx] = g;
}

__global__ void bn_fold_kernel(const float* __restrict__ gamma, const float* __restrict__ beta,
                               const float* __restrict__ mean, const float* __restrict__ var, float eps,
                               float* __restrict__ scale, float* __restrict__ shift, int C, int C_pad) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C_pad) return;
    float s = 0.f, t = 0.f;
    if (c < C) {
        s = gamma[c] / sqrtf(var[c] + eps);
        t = beta[c] - mean[c] * s;
    }
    scale[c] = s; shift[c] = t;
}

// dz = dy * (y > 0); s1[c] += sum dz; s2[c] += sum dz*y.   blockDim = (C, rows)
// ORDERED: the block's sums are stored, not added: s1 / s2 point at column 0 of slot 0 of a [grid][2][C] workspace
// (sci_act_bwd_ordered), block b writes slot b, and sci_ordered_slot_sum adds the slots in slot order.
template <bool ORDERED>
__global__ void act_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ y, float* __restrict__ dz,
                               long n_pix, int C, int relu, float* __restrict__ s1, float* __restrict__ s2) {
    extern __shared__ float sm[];
    const int c = threadIdx.x, row = threadIdx.y, rows = blockDim.y;
    float a1 = 0.f, a2 = 0.f;
    for (long p = (long)blockIdx.x * rows + row; p < n_pix; p += (long)gridDim.x * rows) {
        const long o = p * C + c;
        const float yv = y ? y[o] : 0.f;
        float g = dy[o];
        if (relu && !(yv > 0.f)) g = 0.f;
        dz[o] = g;
        a1 += g; a2 += g * yv;
    }
    if (s1 || s2) {
        sm[(row * C + c) * 2] = a1; sm[(row * C + c) * 2 + 1] = a2;
        __syncthreads();
        if (row == 0) {
            for (int r = 1; r < rows; ++r) { a1 += sm[(r * C + c) * 2]; a2 += sm[(r * C + c) * 2 + 1]; }
            if (ORDERED) {
                const long o = (long)blockIdx.x * 2 * C + c;
                if (s1) s1[o] = a1;
                if (s2) s2[o] = a2;
            } else {
                if (s1) atomicAdd(s1 + c, a1);
                if (s2) atomicAdd(s2 + c, a2);
            }
        }
    }
}

// out0[i] = out0[i] + (((part[0][i] + part[1][i]) + part[2][i]) + ...), strictly in slot order, for i < n; out1 likewise over
// part[b][n + i].  part holds `slots` slots of `width` floats.  blockIdx.y selects the output (NULL outputs are skipped).
// The adds of one output form a chain, so what costs is waiting for its loads: G lanes serve one output, lane j loads slots
// j, j + G, j + 2G, ... (G * K slots in flight per output), and every lane of the group adds the values, broadcast by
// shuffles, in slot order (the group's first lane stores).  G = 32 for few outputs over many slots (column sums: up to
// 2 x 1024 outputs, up to 1184 slots); G = 1 for weight gradients (10^4..10^5 outputs, 24..296 slots), where there are
// threads enough and the shuffles would only add instructions.
template <int G>
__global__ void __launch_bounds__(256) ordered_slot_sum_kernel(const float* __restrict__ part, int slots, long width, long n,
                                                               float* __restrict__ out0, float* __restrict__ out1) {
    constexpr int K = 16;                                  // slots per lane and chunk: a chunk is G * K slots
    const long i = ((long)blockIdx.x * blockDim.x + threadIdx.x) / G;
    const int lane = threadIdx.x % G;
    float* out = blockIdx.y ? out1 : out0;
    const bool active = out != nullptr && i < n;
    const float* pp = part + (blockIdx.y ? n : 0) + (active ? i : 0);
    float s = 0.f;
    for (int b0 = 0; b0 < slots; b0 += G * K) {
        float t[K];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int b = b0 + k * G + lane;
            t[k] = (active && b < slots) ? pp[(long)b * width] : 0.f;
        }
#pragma unroll
        for (int k = 0; k < K; ++k) {
#pragma unroll
            for (int j = 0; j < G; ++j) {
                const float v = G == 1 ? t[k] : __shfl_sync(0xffffffffu, t[k], j, G);
                const int b = b0 + k * G + j;
                if (b == 0) s = v;
                else if (b < slots) s += v;
            }
        }
    }
    if (active && lane == 0) out[i] = out[i] + s;
}

__global__ void bn_param_grad_kernel(const float* __restrict__ s1, const float* __restrict__ s2,
                                     const float* __restrict__ gamma, const float* __restrict__ beta,
                                     float* __restrict__ dgamma, float* __restrict__ dbeta, int C) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    dbeta[c] = s1[c];
    const float g = gamma[c];
    dgamma[c] = (g != 0.f) ? (s2[c] - beta[c] * s1[c]) / g : 0.f;
}

// in [N][2H][2W][C] -> out [N][H][W][4C], column q*C + c, q = dy*2+dx.  One thread moves VEC consecutive channels
// (float4 when C % 4 == 0), grid-stride so that every SM keeps several 16-byte loads in flight.
template <int VEC>
__global__ void __launch_bounds__(256) pixel_unshuffle_kernel(const float* __restrict__ in, float* __restrict__ out, int N, int H,
                                                                int W, int C) {
    const int cv = C / VEC;
    const long total = (long)N * H * W * 4 * cv;
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const int col = (int)(idx % (4 * cv));
        const long p = idx / (4 * cv);
        const int w = (int)(p % W), h = (int)((p / W) % H), n = (int)(p / ((long)W * H));
        const int q = col / cv, c = (col % cv) * VEC;
        const float* src = in + (((long)n * 2 * H + 2 * h + (q >> 1)) * 2 * W + 2 * w + (q & 1)) * C + c;
        float* dst = out + p * 4 * C + (long)q * C + c;
        if (VEC == 4) *reinterpret_cast<float4*>(dst) = ldg_stream4(src);
        else *dst = *src;
    }
}

__global__ void dilate2_kernel(const float* __restrict__ in, float* __restrict__ out, int N, int H, int W, int C) {
    // out [N][2H][2W][C]: out[2h][2w] = in[h][w], zeros elsewhere
    const long total = (long)N * 4 * H * W * C;
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int c = (int)(idx % C);
    const long p = idx / C;
    const int w2 = (int)(p % (2 * W)), h2 = (int)((p / (2 * W)) % (2 * H)), n = (int)(p / (4L * W * H));
    float v = 0.f;
    if (!(w2 & 1) && !(h2 & 1)) v = in[(((long)n * H + (h2 >> 1)) * W + (w2 >> 1)) * C + c];
    out[idx] = v;
}

// ---- FFDNet boundary -----------------------------------------------------------------------------
__device__ __forceinline__ uint4 pack8_h(const __half* v) {
    auto pk = [](__half a, __half b) -> uint32_t { return (uint32_t)__half_as_ushort(a) | ((uint32_t)__half_as_ushort(b) << 16); };
    return make_uint4(pk(v[0], v[1]), pk(v[2], v[3]), pk(v[4], v[5]), pk(v[6], v[7]));
}
__global__ void ffdnet_pack_kernel(const float* __restrict__ u, float sigma, float* __restrict__ out, int B, int C, int H,
                                   int W, int Cpad, int round_tf32) {
    const int h2 = H >> 1, w2 = W >> 1;
    const long total = (long)B * h2 * w2 * Cpad;
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int k = (int)(idx % Cpad);
    const long p = idx / Cpad;
    const int w = (int)(p % w2), h = (int)((p / w2) % h2), n = (int)(p / ((long)w2 * h2));
    // round_tf32: channel k holds tf32(v), channel k+16 the remainder tf32(v - tf32(v)) (weights duplicated)
    const int kk = (round_tf32 && k >= 16) ? k - 16 : k;
    float v = 0.f;
    if (kk < 4 * C) {                                  // KAIR pixel-unshuffle: channel c*4 + dy*2 + dx (basicblock.py:104-126)
        const int c = kk >> 2, dy = (kk >> 1) & 1, dx = kk & 1;
        v = u[(((long)n * C + c) * H + 2 * h + dy) * W + 2 * w + dx];
    } else if (kk == 4 * C) {                          // sigma map appended after the image channels (network_ffdnet.py:63-64)
        v = sigma;
    }
    if (round_tf32) {
        const float hi = rna_tf32(v);
        v = (k >= 16) ? rna_tf32(v - hi) : hi;
    }
    out[idx] = v;
}

// fp16 split form of the same input (inference on conv_fwd2_tc_kernel's `split` path): 64 fp16 channels per pixel,
// channel k < 32 = fp16(v_k), channel 32 + k = fp16((v_k - fp16(v_k)) * 2^11).  One thread per (pixel, 16-byte chunk).
__global__ void ffdnet_pack_split_half_kernel(const float* __restrict__ u, float sigma, __half* __restrict__ out, int B, int C,
                                              int H, int W) {
    const int h2 = H >> 1, w2 = W >> 1;
    const long total = (long)B * h2 * w2 * 8;
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int ch = (int)(idx & 7);                     // 8 channels: ch < 4 -> hi of channels 8ch.., else remainders of 8(ch-4)..
    const long p = idx >> 3;
    const int w = (int)(p % w2), h = (int)((p / w2) % h2), n = (int)(p / ((long)w2 * h2));
    __half r[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int kk = (ch & 3) * 8 + j;
        float v = 0.f;
        if (kk < 4 * C) {
            const int c = kk >> 2, dy = (kk >> 1) & 1, dx = kk & 1;
            v = u[(((long)n * C + c) * H + 2 * h + dy) * W + 2 * w + dx];
        } else if (kk == 4 * C) {
            v = sigma;
        }
        const __half hi = __float2half_rn(v);
        r[j] = (ch < 4) ? hi : __float2half_rn((v - __half2float(hi)) * 2048.f);
    }
    reinterpret_cast<uint4*>(out)[idx] = pack8_h(r);
}

// network output from the split form: y[n][h][w][64] fp16 = [hi 0..31 | remainder * 2^11 0..31] -> xhat planar fp32
__global__ void ffdnet_unpack_split_half_kernel(const __half* __restrict__ y, float* __restrict__ xhat, int B, int C, int H, int W) {
    const long total = (long)B * C * H * W;
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int wf = (int)(idx % W), hf = (int)((idx / W) % H), c = (int)((idx / ((long)W * H)) % C);
    const int n = (int)(idx / ((long)C * W * H));
    const int k = c * 4 + (hf & 1) * 2 + (wf & 1);
    const __half* row = y + (((long)n * (H >> 1) + (hf >> 1)) * (W >> 1) + (wf >> 1)) * 64;
    xhat[idx] = fmaf(__half2float(row[32 + k]), 1.f / 2048.f, __half2float(row[k]));
}

// xhat[n][c][2h+dy][2w+dx] = y[n][h][w][c*4+dy*2+dx]   (nn.PixelShuffle(2), network_ffdnet.py:66)
__global__ void ffdnet_unpack_kernel(const float* __restrict__ y, float* __restrict__ xhat, int B, int C, int H, int W,
                                     int Cpad) {
    const long total = (long)B * C * H * W;
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int wf = (int)(idx % W), hf = (int)((idx / W) % H), c = (int)((idx / ((long)W * H)) % C);
    const int n = (int)(idx / ((long)C * W * H));
    const int k = c * 4 + (hf & 1) * 2 + (wf & 1);
    xhat[idx] = y[(((long)n * (H >> 1) + (hf >> 1)) * (W >> 1) + (wf >> 1)) * Cpad + k];
}

// adjoint: dy[n][h][w][k] = dxhat[n][k>>2][2h+dy][2w+dx] for k < 4C, 0 in the padded columns
__global__ void ffdnet_unpack_grad_kernel(const float* __restrict__ dxhat, float* __restrict__ dy, int B, int C, int H, int W,
                                          int Cpad) {
    const int h2 = H >> 1, w2 = W >> 1;
    const long total = (long)B * h2 * w2 * Cpad;
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int k = (int)(idx % Cpad);
    const long p = idx / Cpad;
    const int w = (int)(p % w2), h = (int)((p / w2) % h2), n = (int)(p / ((long)w2 * h2));
    float v = 0.f;
    if (k < 4 * C) {
        const int c = k >> 2, dy_ = (k >> 1) & 1, dx_ = k & 1;
        v = dxhat[(((long)n * C + c) * H + 2 * h + dy_) * W + 2 * w + dx_];
    }
    dy[idx] = v;
}

// ---- FastDVDnet boundary --------------------------------------------------------------------------
// One thread builds the 32-channel row of one pixel (9 coalesced plane reads), the block transposes it through
// shared memory so that the NHWC write is fully coalesced.
// NC = planes per frame of the planar frames: 3 (colour) or 1 (gray, written as the first plane of the colour layout:
// the other two channels of each slot are +0, exactly what packing the zero-embedded cube gives).
constexpr int FPACK_PIX = 256;
template <int NC>
__global__ void __launch_bounds__(FPACK_PIX) fastdvd_pack_kernel(const float* __restrict__ frames, float sigma,
                                                                   float* __restrict__ out, int B, int H, int W, int Cpad,
                                                                   int round_tf32) {
    extern __shared__ float srow[];                   // [FPACK_PIX][Cpad + 1]
    const long plane = (long)H * W;
    const int f = blockIdx.y;
    const long p0 = (long)blockIdx.x * FPACK_PIX;
    const long p = p0 + threadIdx.x;
    const int CS = Cpad + 1;
    float* row = srow + threadIdx.x * CS;
    for (int k = 0; k < Cpad; ++k) row[k] = 0.f;
    if (p < plane) {
#pragma unroll
        for (int slot = 0; slot < 3; ++slot) {
            const int src = (f + slot - 1 + B) % B;                              // circular window (fastdvdnet.py:115)
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const float v = (c == 3) ? sigma : (c < NC ? frames[((long)src * NC + c) * plane + p] : 0.f);
                if (round_tf32) {        // channel k: tf32(v); channel k+16: remainder (weights duplicated)
                    const float hi = rna_tf32(v);
                    row[slot * 4 + c] = hi;
                    row[16 + slot * 4 + c] = rna_tf32(v - hi);
                } else {
                    row[slot * 4 + c] = v;
                }
            }
        }
    }
    __syncthreads();
    const int npx = (int)min((long)FPACK_PIX, plane - p0);
    float* dst = out + ((long)f * plane + p0) * Cpad;
    for (int i = threadIdx.x; i < npx * Cpad; i += FPACK_PIX) dst[i] = srow[(i / Cpad) * CS + (i % Cpad)];
}

template <int NC>
__global__ void fastdvd_pack_grad_kernel(const float* __restrict__ din, float* __restrict__ dframes, int B, int H, int W,
                                         int Cpad, int accumulate) {
    // dframes[j][c][p] (+)= sum_{slot} din[(j - slot + 1) mod B][p][slot*4 + c], c < NC
    const long plane = (long)H * W;
    const long total = (long)B * NC * plane;
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const long p = idx % plane;
    const int c = (int)((idx / plane) % NC), j = (int)(idx / (NC * plane));
    float v = accumulate ? dframes[idx] : 0.f;
#pragma unroll
    for (int slot = 0; slot < 3; ++slot) {
        const int f = (j - slot + 1 + B) % B;
        v += din[((long)f * plane + p) * Cpad + slot * 4 + c];
    }
    dframes[idx] = v;
}

template <int NC>
__global__ void fastdvd_output_kernel(const float* __restrict__ frames, const float* __restrict__ y, float* __restrict__ out,
                                      int B, int H, int W, int Cpad) {
    const long plane = (long)H * W;
    const long total = (long)B * NC * plane;
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const long p = idx % plane;
    const int c = (int)((idx / plane) % NC), f = (int)(idx / (NC * plane));
    out[idx] = frames[idx] - __ldg(y + ((long)f * plane + p) * Cpad + c);    // models.py:196
}

// dy[f][p][c] = -dout[f][c][p] for c < NC, 0 for the padded columns.  One thread reads the NC plane values of its pixel
// (coalesced), the block writes the [256 px][Cpad] rows through shared memory (fully coalesced NHWC write).
template <int NC>
__global__ void __launch_bounds__(FPACK_PIX) fastdvd_output_grad_kernel(const float* __restrict__ dout, float* __restrict__ dy,
                                                                          int H, int W, int Cpad) {
    extern __shared__ float srow[];                   // [FPACK_PIX][Cpad + 1]
    const long plane = (long)H * W;
    const int f = blockIdx.y;
    const long p0 = (long)blockIdx.x * FPACK_PIX, p = p0 + threadIdx.x;
    const int CS = Cpad + 1;
    float* row = srow + threadIdx.x * CS;
    for (int k = 0; k < Cpad; ++k) row[k] = 0.f;
    if (p < plane) {
#pragma unroll
        for (int c = 0; c < NC; ++c) row[c] = -dout[((long)f * NC + c) * plane + p];
        // gray frames: what the colour kernel writes for the zero planes of the embedded cube, -(+0), so that the backward
        // pass of a gray sequence is bit for bit that of its embedding
        if (NC == 1) row[1] = row[2] = -0.f;
    }
    __syncthreads();
    const int npx = (int)min((long)FPACK_PIX, plane - p0);
    float* dst = dy + ((long)f * plane + p0) * Cpad;
    for (int i = threadIdx.x; i < npx * Cpad; i += FPACK_PIX) dst[i] = srow[(i / Cpad) * CS + (i % Cpad)];
}

__global__ void noisy_input_kernel(const float* __restrict__ v, const double* __restrict__ noise, float* __restrict__ vplus,
                                   long n) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float o = (float)((double)v[i] + noise[i]);      // float32(meas + noise), utils_image.py:188-192
    vplus[i] = v[i] + o;                                    // test_fastdvdnet.py:359
}

// ---- measurement loss -------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) meas_loss_kernel(const float* __restrict__ xhat, const float* __restrict__ phi,
                                                         const float* __restrict__ y, float* __restrict__ dxhat,
                                                         double* __restrict__ loss, int H, int W, int B, int C, float norm,
                                                         double inv_count) {
    __shared__ double red[32];
    const long plane = (long)H * W;
    const long p = (long)blockIdx.x * blockDim.x + threadIdx.x;
    double err = 0.0;
    if (p < plane) {
        const int row = (int)(p / W), col = (int)(p % W);
        const int c = (C == 3) ? (row & 1) + (col & 1) : 0;       // colour: RGGB sample; gray: the pixel itself
        float up = 0.f;
        for (int t = 0; t < B; ++t) up += xhat[((long)t * C + c) * plane + p] * phi[t * plane + p];
        const float diff = up - y[p];
        err = (double)(diff * diff);
        if (dxhat) {
            const float g = norm * diff;                      // mse_loss backward: (2/N) * (input - target)
            for (int t = 0; t < B; ++t) {
                const float gv = g * phi[t * plane + p];
                for (int k = 0; k < C; ++k) dxhat[((long)t * C + k) * plane + p] = (k == c) ? gv : 0.f;
            }
        }
    }
    const double s = block_sum(err, red);
    if (threadIdx.x == 0) atomicAdd(loss, s * inv_count);
}

__global__ void adam_kernel(float* __restrict__ param, const float* __restrict__ grad, float* __restrict__ m,
                            float* __restrict__ v, long n, float one_m_beta1, float beta2, float one_m_beta2, float eps,
                            float step_size, float bc2_sqrt) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float g = grad[i];
    float mi = m[i], vi = v[i];
    mi = mi + one_m_beta1 * (g - mi);                       // exp_avg.lerp_(grad, 1-beta1)
    vi = vi * beta2 + one_m_beta2 * (g * g);                // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1-beta2)
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    param[i] = param[i] - step_size * (mi / denom);         // param.addcdiv_(exp_avg, denom, value=-step_size)
    m[i] = mi; v[i] = vi;
}

inline int grid1d(long n, int block = 256) { return (int)((n + block - 1) / block); }

}  // namespace

// ---- fp16 forms (inference chains on the kind::f16 tensor-core kernels) ---------------------------------------------
// packed[tap][col][k] as IEEE binary16 (round to nearest), forward form only.  Same column / dup rules as above.
__global__ void pack_weights_half_kernel(const float* __restrict__ w, __half* __restrict__ packed, int Co, int Ci, int groups,
                                         int Co_pad, int Ci_pad, int ps, int ci_dup) {
    const long total = (long)9 * Co_pad * Ci_pad;
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    int ci = (int)(idx % Ci_pad);
    const int col = (int)((idx / Ci_pad) % Co_pad), tap = (int)(idx / ((long)Ci_pad * Co_pad));
    float v = 0.f;
    if (ci_dup > 0 && ci >= ci_dup && ci < ci_dup + Ci) ci -= ci_dup;
    // ci_dup == -1: split form (conv_fwd2_tc_kernel, `split`): K chunk g of 64 = [fp16(w) of channels 32g..32g+31 | the
    // remainders (w - fp16(w)) * 2^11 of the same channels]
    const int part = (ci_dup == -1) ? (ci >> 5) & 1 : 0;
    if (ci_dup == -1) ci = ((ci >> 6) << 5) | (ci & 31);
    const int q = Co_pad >> 2;
    const int co = ps ? (col % q) * 4 + col / q : col;
    if ((ps ? (col % q) < (Co >> 2) : col < Co) && ci < Ci) {
        const int cig = Ci / groups, cog = Co / groups, g = co / cog;
        if (ci / cig == g) v = w[((long)co * cig + (ci - g * cig)) * 9 + tap];
    }
    if (part) v = (v - __half2float(__float2half_rn(v))) * 2048.f;
    packed[idx] = __float2half_rn(v);
}

// FastDVDnet input block as fp16 NHWC rows of 64 channels (128 bytes): channel k = fp16(v), channel k + 16 = fp16(v - fp16(v))
// (the first layer's weights are duplicated there, ci_dup = 16), everything else zero.  One thread per pixel, eight
// 16-byte stores = one full 128-byte line.
__device__ __forceinline__ uint4 pack8(const __half* v) {
    auto pk = [](__half a, __half b) -> uint32_t { return (uint32_t)__half_as_ushort(a) | ((uint32_t)__half_as_ushort(b) << 16); };
    return make_uint4(pk(v[0], v[1]), pk(v[2], v[3]), pk(v[4], v[5]), pk(v[6], v[7]));
}
// NCH = 16-byte chunks per pixel row: 8 (64 channels, the upper 36 zero) or 4 (32 channels = 64-byte rows); NC = planes per
// frame as in fastdvd_pack_kernel
template <int NCH, int NC>
__global__ void __launch_bounds__(256) fastdvd_pack_half_kernel(const float* __restrict__ frames, float sigma,
                                                                __half* __restrict__ out, int B, int H, int W) {
    __shared__ uint4 tile[8][32 * NCH];               // per warp: 32 pixels x NCH chunks of 16 bytes, XOR-swizzled
    const long plane = (long)H * W;
    const int f = blockIdx.y;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long p0 = (long)blockIdx.x * blockDim.x + warp * 32;       // first pixel of this warp
    const long p = p0 + lane;
    __half hi[16], lo[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) { hi[k] = __float2half_rn(0.f); lo[k] = hi[k]; }
    if (p < plane) {
#pragma unroll
        for (int slot = 0; slot < 3; ++slot) {
            const int src = (f + slot - 1 + B) % B;                          // circular window (fastdvdnet.py:115)
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const float v = (c == 3) ? sigma : (c < NC ? __ldg(frames + ((long)src * NC + c) * plane + p) : 0.f);
                const __half h = __float2half_rn(v);
                hi[slot * 4 + c] = h;
                lo[slot * 4 + c] = __float2half_rn(v - __half2float(h));
            }
        }
    }
    // stage the warp's 32 pixel rows (chunk j of pixel l at slot l*NCH + (j ^ (l & (NCH-1))): conflict-free both ways) ...
    uint4* t = tile[warp];
    const uint4 z = make_uint4(0u, 0u, 0u, 0u);
    const int sw = lane & (NCH - 1);
    t[lane * NCH + (0 ^ sw)] = pack8(hi);
    t[lane * NCH + (1 ^ sw)] = pack8(hi + 8);
    t[lane * NCH + (2 ^ sw)] = pack8(lo);
    t[lane * NCH + (3 ^ sw)] = pack8(lo + 8);
#pragma unroll
    for (int j = 4; j < NCH; ++j) t[lane * NCH + (j ^ sw)] = z;
    __syncwarp();
    // ... and write them as fully coalesced 512-byte warp stores
    uint4* dst = reinterpret_cast<uint4*>(out + ((long)f * plane + p0) * (NCH * 8));
#pragma unroll
    for (int i = 0; i < NCH; ++i) {
        const int o = i * 32 + lane, px = o / NCH, j = o % NCH;
        if (p0 + px < plane) dst[o] = t[px * NCH + (j ^ (px & (NCH - 1)))];
    }
}

// ---- batched per-layer bookkeeping ------------------------------------------------------------------------------------
// A fine-tune step used to issue ~250 launches of 3-4 us each (weight (re)packing, BatchNorm folding, gradient unpacking,
// BatchNorm parameter gradients: one launch per layer and kind).  The engine now keeps a device-side table of these
// operations (pointers are stable: parameters live in one flat bucket) and runs a whole phase as ONE launch:
// blockIdx.y selects the table entry, blockIdx.x the 256-element slice of it.
__device__ __forceinline__ void layer_op_element(const sci_layer_op& d, long idx) {
    switch (d.kind) {
    case 0: {   // pack_weights (forward or transposed / flipped data-gradient form), see pack_weights_kernel
        const long total = (long)9 * d.Co_pad * d.Ci_pad;
        if (idx >= total) return;
        const float* w = static_cast<const float*>(d.a);
        const float* oscale = static_cast<const float*>(d.b);
        float* packed = static_cast<float*>(d.o0);
        int tap, col, ci;
        if (!d.tflip) { ci = (int)(idx % d.Ci_pad); col = (int)((idx / d.Ci_pad) % d.Co_pad); tap = (int)(idx / ((long)d.Ci_pad * d.Co_pad)); }
        else          { col = (int)(idx % d.Co_pad); ci = (int)((idx / d.Co_pad) % d.Ci_pad); tap = (int)(idx / ((long)d.Ci_pad * d.Co_pad)); }
        float v = 0.f;
        if (d.ci_dup > 0 && ci >= d.ci_dup && ci < d.ci_dup + d.Ci) ci -= d.ci_dup;
        const int q = d.Co_pad >> 2;
        const int co = d.ps ? (col % q) * 4 + col / q : col;
        if ((d.ps ? (col % q) < (d.Co >> 2) : col < d.Co) && ci < d.Ci) {
            const int cig = d.Ci / d.groups, cog = d.Co / d.groups, g = co / cog;
            if (ci / cig == g) {
                v = w[((long)co * cig + (ci - g * cig)) * 9 + (d.tflip ? 8 - tap : tap)];
                if (d.tflip && oscale) v = v * oscale[col];
            }
        }
        if (d.round_tf32 == 2) {
            const float hi = rna_tf32(v);
            packed[idx] = hi;
            packed[idx + total] = rna_tf32(v - hi);
            return;
        }
        packed[idx] = d.round_tf32 ? rna_tf32(v) : v;
        return;
    }
    case 1: {   // pack_weights_s2t
        const long total = (long)9 * 4 * d.Ci_pad * d.Co_pad;
        if (idx >= total) return;
        const float* w = static_cast<const float*>(d.a);
        const float* oscale = static_cast<const float*>(d.b);
        const int co = (int)(idx % d.Co_pad);
        const int col = (int)((idx / d.Co_pad) % (4 * d.Ci_pad));
        const int tap = (int)(idx / ((long)d.Co_pad * 4 * d.Ci_pad));
        const int q = col / d.Ci_pad, ci = col % d.Ci_pad;
        const int kh = s2t_src_tap(q >> 1, tap / 3 - 1), kw = s2t_src_tap(q & 1, tap % 3 - 1);
        float v = 0.f;
        if (co < d.Co && ci < d.Ci && kh >= 0 && kw >= 0) {
            v = w[((long)co * d.Ci + ci) * 9 + kh * 3 + kw];
            if (oscale) v = v * oscale[co];
        }
        static_cast<float*>(d.o0)[idx] = d.round_tf32 ? rna_tf32(v) : v;
        return;
    }
    case 2: {   // pack_weights_half
        const long total = (long)9 * d.Co_pad * d.Ci_pad;
        if (idx >= total) return;
        const float* w = static_cast<const float*>(d.a);
        int ci = (int)(idx % d.Ci_pad);
        const int col = (int)((idx / d.Ci_pad) % d.Co_pad), tap = (int)(idx / ((long)d.Ci_pad * d.Co_pad));
        float v = 0.f;
        if (d.ci_dup > 0 && ci >= d.ci_dup && ci < d.ci_dup + d.Ci) ci -= d.ci_dup;
        const int part = (d.ci_dup == -1) ? (ci >> 5) & 1 : 0;      // split form, see pack_weights_half_kernel
        if (d.ci_dup == -1) ci = ((ci >> 6) << 5) | (ci & 31);
        const int q = d.Co_pad >> 2;
        const int co = d.ps ? (col % q) * 4 + col / q : col;
        if ((d.ps ? (col % q) < (d.Co >> 2) : col < d.Co) && ci < d.Ci) {
            const int cig = d.Ci / d.groups, cog = d.Co / d.groups, g = co / cog;
            if (ci / cig == g) v = w[((long)co * cig + (ci - g * cig)) * 9 + tap];
        }
        if (part) v = (v - __half2float(__float2half_rn(v))) * 2048.f;
        static_cast<__half*>(d.o0)[idx] = __float2half_rn(v);
        return;
    }
    case 3: {   // unpack_wgrad
        const int cig = d.Ci / d.groups, cog = d.Co / d.groups;
        if (idx >= (long)d.Co * cig * 9) return;
        const float* packed = static_cast<const float*>(d.a);
        const int tap = (int)(idx % 9), cil = (int)((idx / 9) % cig), co = (int)(idx / (9L * cig));
        const int ci = (co / cog) * cig + cil;
        const int col = out_column(co, d.Co_pad, d.ps);
        float g = packed[((long)tap * d.Co_pad + col) * d.Ci_pad + ci];
        if (d.ci_dup > 0) g += packed[((long)tap * d.Co_pad + col) * d.Ci_pad + ci + d.ci_dup];
        static_cast<float*>(d.o0)[idx] = g;
        return;
    }
    case 4: {   // bn_fold: a gamma, b beta, c mean, d var -> o0 scale, o1 shift (Co real of Co_pad columns)
        if (idx >= d.Co_pad) return;
        float sc = 0.f, sh = 0.f;
        if (idx < d.Co) {
            sc = static_cast<const float*>(d.a)[idx] / sqrtf(static_cast<const float*>(d.d)[idx] + d.eps);
            sh = static_cast<const float*>(d.b)[idx] - static_cast<const float*>(d.c)[idx] * sc;
        }
        static_cast<float*>(d.o0)[idx] = sc;
        static_cast<float*>(d.o1)[idx] = sh;
        return;
    }
    case 5: {   // bn_param_grad: a s1, b s2, c gamma, d beta -> o0 dgamma, o1 dbeta
        if (idx >= d.Co) return;
        const float s1 = static_cast<const float*>(d.a)[idx], g = static_cast<const float*>(d.c)[idx];
        static_cast<float*>(d.o1)[idx] = s1;
        static_cast<float*>(d.o0)[idx] = (g != 0.f) ? (static_cast<const float*>(d.b)[idx] - static_cast<const float*>(d.d)[idx] * s1) / g : 0.f;
        return;
    }
    case 6:     // copy Co floats (bias -> shift column vector, column sums -> bias gradient)
        if (idx < d.Co) static_cast<float*>(d.o0)[idx] = static_cast<const float*>(d.a)[idx];
        return;
    default:
        return;
    }
}

__global__ void __launch_bounds__(256) layer_ops_batch_kernel(const sci_layer_op* __restrict__ table) {
    const sci_layer_op d = table[blockIdx.y];
    layer_op_element(d, (long)blockIdx.x * blockDim.x + threadIdx.x);
}

extern "C" int sci_layer_ops_batch(const sci_layer_op* table_device, int n_ops, int max_blocks, void* stream) {
    SCI_REQUIRE(table_device && n_ops > 0 && n_ops <= 65535 && max_blocks > 0, "layer_ops_batch");
    layer_ops_batch_kernel<<<dim3(max_blocks, n_ops), 256, 0, sci_stream(stream)>>>(table_device);
    SCI_CHECK_LAUNCH("layer_ops_batch");
    return SCI_OK;
}

extern "C" int sci_conv_pack_weights(const float* w, float* packed, int Co, int Ci, int groups, int Co_pad, int Ci_pad,
                                     int ps, const float* oscale, int transpose_flip, int round_tf32, int ci_dup,
                                     void* stream) {
    SCI_REQUIRE(w && packed && Co > 0 && Ci > 0 && groups > 0 && Co % groups == 0 && Ci % groups == 0, "pack_weights");
    SCI_REQUIRE(Co_pad >= Co && Ci_pad >= Ci && (!ps || Co % 4 == 0), "pack_weights: padding / pixel-shuffle");
    SCI_REQUIRE(!ps || Co_pad % 4 == 0, "pack_weights: pixel-shuffle needs Co_pad % 4 == 0");
    SCI_REQUIRE(ci_dup == 0 || (ci_dup >= Ci && ci_dup + Ci <= Ci_pad), "pack_weights: ci_dup block does not fit");
    SCI_REQUIRE(round_tf32 != 2 || !transpose_flip, "pack_weights: split form is for forward weights only");
    const long total = (long)9 * Co_pad * Ci_pad;
    pack_weights_kernel<<<grid1d(total), 256, 0, sci_stream(stream)>>>(w, packed, Co, Ci, groups, Co_pad, Ci_pad, ps, oscale,
                                                                       transpose_flip, round_tf32, ci_dup);
    SCI_CHECK_LAUNCH("pack_weights");
    return SCI_OK;
}

extern "C" int sci_conv_pack_weights_half(const float* w, void* packed, int Co, int Ci, int groups, int Co_pad, int Ci_pad,
                                          int ps, int ci_dup, void* stream) {
    SCI_REQUIRE(w && packed && Co > 0 && Ci > 0 && groups > 0 && Co % groups == 0 && Ci % groups == 0, "pack_weights_half");
    SCI_REQUIRE(Co_pad >= Co && Ci_pad >= Ci && Ci_pad % 32 == 0 && (!ps || (Co % 4 == 0 && Co_pad % 4 == 0)), "pack_weights_half: padding");
    SCI_REQUIRE(ci_dup == 0 || (ci_dup == -1 && Ci_pad % 64 == 0 && Ci_pad >= 2 * ((Ci + 31) / 32) * 32) || (ci_dup >= Ci && ci_dup + Ci <= Ci_pad),
                "pack_weights_half: ci_dup block does not fit");
    const long total = (long)9 * Co_pad * Ci_pad;
    pack_weights_half_kernel<<<grid1d(total), 256, 0, sci_stream(stream)>>>(w, reinterpret_cast<__half*>(packed), Co, Ci, groups,
                                                                            Co_pad, Ci_pad, ps, ci_dup);
    SCI_CHECK_LAUNCH("pack_weights_half");
    return SCI_OK;
}

extern "C" int sci_fastdvd_pack_input_half_planes(const float* frames, float sigma, void* out, int B, int NC, int H, int W, int C,
                                                  void* stream) {
    SCI_REQUIRE(frames && out && B > 0 && H > 0 && W > 0 && B <= 65535 && (C == 32 || C == 64) && (NC == 1 || NC == 3),
                "fastdvd_pack_input_half");
    const dim3 grid(grid1d((long)H * W, 256), B);
    __half* o = reinterpret_cast<__half*>(out);
    if (NC == 3) {
        if (C == 64) fastdvd_pack_half_kernel<8, 3><<<grid, 256, 0, sci_stream(stream)>>>(frames, sigma, o, B, H, W);
        else         fastdvd_pack_half_kernel<4, 3><<<grid, 256, 0, sci_stream(stream)>>>(frames, sigma, o, B, H, W);
    } else {
        if (C == 64) fastdvd_pack_half_kernel<8, 1><<<grid, 256, 0, sci_stream(stream)>>>(frames, sigma, o, B, H, W);
        else         fastdvd_pack_half_kernel<4, 1><<<grid, 256, 0, sci_stream(stream)>>>(frames, sigma, o, B, H, W);
    }
    SCI_CHECK_LAUNCH("fastdvd_pack_input_half");
    return SCI_OK;
}

extern "C" int sci_fastdvd_pack_input_half(const float* frames, float sigma, void* out, int B, int H, int W, int C, void* stream) {
    return sci_fastdvd_pack_input_half_planes(frames, sigma, out, B, 3, H, W, C, stream);
}

extern "C" int sci_conv_pack_weights_s2t(const float* w, float* packed, int Co, int Ci, int Co_pad, int Ci_pad,
                                         const float* oscale, int round_tf32, void* stream) {
    SCI_REQUIRE(w && packed && Co > 0 && Ci > 0 && Co_pad >= Co && Ci_pad >= Ci, "pack_weights_s2t");
    const long total = (long)9 * 4 * Ci_pad * Co_pad;
    pack_weights_s2t_kernel<<<grid1d(total), 256, 0, sci_stream(stream)>>>(w, packed, Co, Ci, Co_pad, Ci_pad, oscale, round_tf32);
    SCI_CHECK_LAUNCH("pack_weights_s2t");
    return SCI_OK;
}

extern "C" int sci_conv_unpack_wgrad(const float* packed_dw, float* dw, int Co, int Ci, int groups, int Co_pad, int Ci_pad,
                                     int ps, int ci_dup, void* stream) {
    SCI_REQUIRE(packed_dw && dw && Co > 0 && Ci > 0 && groups > 0 && Co_pad >= Co && Ci_pad >= Ci, "unpack_wgrad");
    SCI_REQUIRE(ci_dup == 0 || (ci_dup >= Ci && ci_dup + Ci <= Ci_pad), "unpack_wgrad: ci_dup block does not fit");
    const long total = (long)Co * (Ci / groups) * 9;
    unpack_wgrad_kernel<<<grid1d(total), 256, 0, sci_stream(stream)>>>(packed_dw, dw, Co, Ci, groups, Co_pad, Ci_pad, ps,
                                                                       ci_dup);
    SCI_CHECK_LAUNCH("unpack_wgrad");
    return SCI_OK;
}

extern "C" int sci_bn_fold(const float* gamma, const float* beta, const float* mean, const float* var, float eps,
                           float* scale, float* shift, int C, int C_pad, void* stream) {
    SCI_REQUIRE(gamma && beta && mean && var && scale && shift && C > 0 && C_pad >= C, "bn_fold");
    bn_fold_kernel<<<grid1d(C_pad, 128), 128, 0, sci_stream(stream)>>>(gamma, beta, mean, var, eps, scale, shift, C, C_pad);
    SCI_CHECK_LAUNCH("bn_fold");
    return SCI_OK;
}

int sci_ordered_slot_sum(const float* part, int slots, long width, long n, float* out0, float* out1, void* stream) {
    if (!out0 && !out1) return SCI_OK;
    const dim3 block(256);
    if (n <= 2048)
        ordered_slot_sum_kernel<32><<<dim3(grid1d(32 * n), out1 ? 2 : 1), block, 0, sci_stream(stream)>>>(part, slots, width, n,
                                                                                                          out0, out1);
    else
        ordered_slot_sum_kernel<1><<<dim3(grid1d(n), out1 ? 2 : 1), block, 0, sci_stream(stream)>>>(part, slots, width, n, out0,
                                                                                                    out1);
    SCI_CHECK_LAUNCH("ordered slot sum");
    return SCI_OK;
}

namespace {
// launch shape of act_bwd_kernel: blocks of (C, rows) threads, at most 8 per SM
int act_bwd_rows(int C) { return max(1, 256 / C); }
int act_bwd_grid(long n_pix, int C) { return (int)min((long)SCI_NUM_SMS * 8, (n_pix + act_bwd_rows(C) - 1) / act_bwd_rows(C)); }

int act_bwd_launch(bool ordered, const float* dy, const float* y, float* dz, long n_pix, int C, int relu, float* s1, float* s2,
                   void* stream) {
    const int rows = act_bwd_rows(C);
    const dim3 block(C, rows);
    const int grid = act_bwd_grid(n_pix, C);
    const size_t smem = (size_t)rows * C * 2 * sizeof(float);
    (ordered ? act_bwd_kernel<true> : act_bwd_kernel<false>)<<<grid, block, smem, sci_stream(stream)>>>(dy, y, dz, n_pix, C,
                                                                                                         relu, s1, s2);
    SCI_CHECK_LAUNCH("act_bwd");
    return SCI_OK;
}
}  // namespace

extern "C" int sci_act_bwd(const float* dy, const float* y, float* dz, long n_pix, int C, int relu, float* s1, float* s2,
                           void* stream) {
    SCI_REQUIRE(dy && dz && n_pix > 0 && C > 0 && C <= 1024, "act_bwd");
    SCI_REQUIRE(!(relu || s2) || y, "act_bwd: y needed for relu / s2");
    return act_bwd_launch(false, dy, y, dz, n_pix, C, relu, s1, s2, stream);
}

extern "C" size_t sci_act_bwd_workspace_bytes(long n_pix, int C) {
    if (n_pix <= 0 || C <= 0 || C > 1024) return 0;
    return (size_t)act_bwd_grid(n_pix, C) * 2 * C * sizeof(float);
}

extern "C" int sci_act_bwd_ordered(const float* dy, const float* y, float* dz, long n_pix, int C, int relu, float* s1,
                                   float* s2, void* workspace, size_t workspace_bytes, void* stream) {
    SCI_REQUIRE(dy && dz && n_pix > 0 && C > 0 && C <= 1024, "act_bwd");
    SCI_REQUIRE(!(relu || s2) || y, "act_bwd: y needed for relu / s2");
    SCI_REQUIRE(workspace && workspace_bytes >= sci_act_bwd_workspace_bytes(n_pix, C), "act_bwd ordered: workspace missing or too small");
    SCI_REQUIRE(((uintptr_t)workspace & 15) == 0, "act_bwd ordered: workspace must be 16-byte aligned");
    float* ws = static_cast<float*>(workspace);
    int rc = act_bwd_launch(true, dy, y, dz, n_pix, C, relu, s1 ? ws : nullptr, s2 ? ws + C : nullptr, stream);
    if (rc) return rc;
    return sci_ordered_slot_sum(ws, act_bwd_grid(n_pix, C), 2L * C, C, s1, s2, stream);
}

extern "C" int sci_bn_param_grad(const float* s1, const float* s2, const float* gamma, const float* beta, float* dgamma,
                                 float* dbeta, int C, void* stream) {
    SCI_REQUIRE(s1 && s2 && gamma && beta && dgamma && dbeta && C > 0, "bn_param_grad");
    bn_param_grad_kernel<<<grid1d(C, 128), 128, 0, sci_stream(stream)>>>(s1, s2, gamma, beta, dgamma, dbeta, C);
    SCI_CHECK_LAUNCH("bn_param_grad");
    return SCI_OK;
}

extern "C" int sci_nhwc_pixel_unshuffle(const float* in, float* out, int N, int H, int W, int C, void* stream) {
    SCI_REQUIRE(in && out && N > 0 && H > 0 && W > 0 && C > 0, "pixel_unshuffle");
    const bool v4 = C % 4 == 0 && (((uintptr_t)in | (uintptr_t)out) & 15) == 0;
    const long work = (long)N * H * W * 4 * (v4 ? C / 4 : C);
    const int grid = (int)min((long)SCI_NUM_SMS * 16, (work + 255) / 256);
    if (v4) pixel_unshuffle_kernel<4><<<grid, 256, 0, sci_stream(stream)>>>(in, out, N, H, W, C);
    else    pixel_unshuffle_kernel<1><<<grid, 256, 0, sci_stream(stream)>>>(in, out, N, H, W, C);
    SCI_CHECK_LAUNCH("pixel_unshuffle");
    return SCI_OK;
}

extern "C" int sci_nhwc_dilate2(const float* in, float* out, int N, int H, int W, int C, void* stream) {
    SCI_REQUIRE(in && out && N > 0 && H > 0 && W > 0 && C > 0, "dilate2");
    dilate2_kernel<<<grid1d((long)N * 4 * H * W * C), 256, 0, sci_stream(stream)>>>(in, out, N, H, W, C);
    SCI_CHECK_LAUNCH("dilate2");
    return SCI_OK;
}

extern "C" int sci_ffdnet_pack_input(const float* u, float sigma, float* out, int B, int C, int H, int W, int Cpad,
                                     int round_tf32, void* stream) {
    SCI_REQUIRE(u && out && B > 0 && (C == 1 || C == 3) && H > 0 && W > 0 && H % 2 == 0 && W % 2 == 0 &&
                Cpad >= (round_tf32 ? 32 : 4 * C + 1), "ffdnet_pack_input");
    ffdnet_pack_kernel<<<grid1d((long)B * (H / 2) * (W / 2) * Cpad), 256, 0, sci_stream(stream)>>>(u, sigma, out, B, C, H, W,
                                                                                                 Cpad, round_tf32);
    SCI_CHECK_LAUNCH("ffdnet_pack_input");
    return SCI_OK;
}

extern "C" int sci_ffdnet_unpack_output(const float* y, float* xhat, int B, int C, int H, int W, int Cpad, void* stream) {
    SCI_REQUIRE(y && xhat && B > 0 && (C == 1 || C == 3) && H % 2 == 0 && W % 2 == 0 && Cpad >= 4 * C, "ffdnet_unpack_output");
    ffdnet_unpack_kernel<<<grid1d((long)B * C * H * W), 256, 0, sci_stream(stream)>>>(y, xhat, B, C, H, W, Cpad);
    SCI_CHECK_LAUNCH("ffdnet_unpack_output");
    return SCI_OK;
}

extern "C" int sci_ffdnet_pack_input_split_half(const float* u, float sigma, void* out, int B, int C, int H, int W, void* stream) {
    SCI_REQUIRE(u && out && B > 0 && (C == 1 || C == 3) && H > 0 && W > 0 && H % 2 == 0 && W % 2 == 0, "ffdnet_pack_input_split_half");
    ffdnet_pack_split_half_kernel<<<grid1d((long)B * (H / 2) * (W / 2) * 8), 256, 0, sci_stream(stream)>>>(
        u, sigma, reinterpret_cast<__half*>(out), B, C, H, W);
    SCI_CHECK_LAUNCH("ffdnet_pack_input_split_half");
    return SCI_OK;
}

extern "C" int sci_ffdnet_unpack_output_split_half(const void* y, float* xhat, int B, int C, int H, int W, void* stream) {
    SCI_REQUIRE(y && xhat && B > 0 && (C == 1 || C == 3) && H % 2 == 0 && W % 2 == 0, "ffdnet_unpack_output_split_half");
    ffdnet_unpack_split_half_kernel<<<grid1d((long)B * C * H * W), 256, 0, sci_stream(stream)>>>(
        reinterpret_cast<const __half*>(y), xhat, B, C, H, W);
    SCI_CHECK_LAUNCH("ffdnet_unpack_output_split_half");
    return SCI_OK;
}

extern "C" int sci_ffdnet_unpack_output_grad(const float* dxhat, float* dy, int B, int C, int H, int W, int Cpad,
                                             void* stream) {
    SCI_REQUIRE(dy && dxhat && B > 0 && (C == 1 || C == 3) && H % 2 == 0 && W % 2 == 0 && Cpad >= 4 * C,
                "ffdnet_unpack_output_grad");
    ffdnet_unpack_grad_kernel<<<grid1d((long)B * (H / 2) * (W / 2) * Cpad), 256, 0, sci_stream(stream)>>>(dxhat, dy, B, C, H,
                                                                                                          W, Cpad);
    SCI_CHECK_LAUNCH("ffdnet_unpack_output_grad");
    return SCI_OK;
}

extern "C" int sci_fastdvd_pack_input_planes(const float* frames, float sigma, float* out, int B, int NC, int H, int W, int Cpad,
                                             int round_tf32, void* stream) {
    SCI_REQUIRE(frames && out && B > 0 && H > 0 && W > 0 && Cpad >= (round_tf32 ? 32 : 12) && (NC == 1 || NC == 3),
                "fastdvd_pack_input");
    SCI_REQUIRE(Cpad <= 48 && B <= 65535, "fastdvd_pack_input: Cpad <= 48");
    const size_t smem = (size_t)FPACK_PIX * (Cpad + 1) * sizeof(float);
    // the largest Cpad admitted above, so that the once-per-device limit covers every later call
    const void* kern = NC == 3 ? (const void*)fastdvd_pack_kernel<3> : (const void*)fastdvd_pack_kernel<1>;
    const cudaError_t e = sci_smem_limit(kern, FPACK_PIX * (48 + 1) * (int)sizeof(float));
    if (e != cudaSuccess) return sci_fail(SCI_ELAUNCH, "fastdvd_pack_input: shared-memory limit", e);
    const dim3 grid(grid1d((long)H * W, FPACK_PIX), B);
    if (NC == 3) fastdvd_pack_kernel<3><<<grid, FPACK_PIX, smem, sci_stream(stream)>>>(frames, sigma, out, B, H, W, Cpad, round_tf32);
    else         fastdvd_pack_kernel<1><<<grid, FPACK_PIX, smem, sci_stream(stream)>>>(frames, sigma, out, B, H, W, Cpad, round_tf32);
    SCI_CHECK_LAUNCH("fastdvd_pack_input");
    return SCI_OK;
}

extern "C" int sci_fastdvd_pack_input(const float* frames, float sigma, float* out, int B, int H, int W, int Cpad,
                                      int round_tf32, void* stream) {
    return sci_fastdvd_pack_input_planes(frames, sigma, out, B, 3, H, W, Cpad, round_tf32, stream);
}

extern "C" int sci_fastdvd_pack_input_grad_planes(const float* din, float* dframes, int B, int NC, int H, int W, int Cpad,
                                                  int accumulate, void* stream) {
    SCI_REQUIRE(din && dframes && B > 0 && H > 0 && W > 0 && Cpad >= 12 && (NC == 1 || NC == 3), "fastdvd_pack_input_grad");
    const int grid = grid1d((long)B * NC * H * W);
    if (NC == 3) fastdvd_pack_grad_kernel<3><<<grid, 256, 0, sci_stream(stream)>>>(din, dframes, B, H, W, Cpad, accumulate);
    else         fastdvd_pack_grad_kernel<1><<<grid, 256, 0, sci_stream(stream)>>>(din, dframes, B, H, W, Cpad, accumulate);
    SCI_CHECK_LAUNCH("fastdvd_pack_input_grad");
    return SCI_OK;
}

extern "C" int sci_fastdvd_pack_input_grad(const float* din, float* dframes, int B, int H, int W, int Cpad, int accumulate,
                                           void* stream) {
    return sci_fastdvd_pack_input_grad_planes(din, dframes, B, 3, H, W, Cpad, accumulate, stream);
}

extern "C" int sci_fastdvd_output_planes(const float* frames, const float* y, float* out, int B, int NC, int H, int W, int Cpad,
                                         void* stream) {
    SCI_REQUIRE(frames && y && out && B > 0 && H > 0 && W > 0 && (NC == 1 || NC == 3) && Cpad >= NC, "fastdvd_output");
    const int grid = grid1d((long)B * NC * H * W);
    if (NC == 3) fastdvd_output_kernel<3><<<grid, 256, 0, sci_stream(stream)>>>(frames, y, out, B, H, W, Cpad);
    else         fastdvd_output_kernel<1><<<grid, 256, 0, sci_stream(stream)>>>(frames, y, out, B, H, W, Cpad);
    SCI_CHECK_LAUNCH("fastdvd_output");
    return SCI_OK;
}

extern "C" int sci_fastdvd_output(const float* frames, const float* y, float* out, int B, int H, int W, int Cpad,
                                  void* stream) {
    return sci_fastdvd_output_planes(frames, y, out, B, 3, H, W, Cpad, stream);
}

extern "C" int sci_fastdvd_output_grad_planes(const float* dout, float* dy, int B, int NC, int H, int W, int Cpad, void* stream) {
    SCI_REQUIRE(dout && dy && B > 0 && H > 0 && W > 0 && (NC == 1 || NC == 3) && Cpad >= NC, "fastdvd_output_grad");
    SCI_REQUIRE(Cpad <= 64, "fastdvd_output_grad: Cpad");
    // 256 * (Cpad + 1) floats pass the 48 KB default from Cpad 48 on; raise the limit to what Cpad 64 needs
    const void* kern = NC == 3 ? (const void*)fastdvd_output_grad_kernel<3> : (const void*)fastdvd_output_grad_kernel<1>;
    const cudaError_t e = sci_smem_limit(kern, FPACK_PIX * (64 + 1) * (int)sizeof(float));
    if (e != cudaSuccess) return sci_fail(SCI_ELAUNCH, "fastdvd_output_grad: shared-memory limit", e);
    const long plane = (long)H * W;
    const dim3 grid(grid1d(plane, FPACK_PIX), B);
    const size_t smem = (size_t)FPACK_PIX * (Cpad + 1) * sizeof(float);
    if (NC == 3) fastdvd_output_grad_kernel<3><<<grid, FPACK_PIX, smem, sci_stream(stream)>>>(dout, dy, H, W, Cpad);
    else         fastdvd_output_grad_kernel<1><<<grid, FPACK_PIX, smem, sci_stream(stream)>>>(dout, dy, H, W, Cpad);
    SCI_CHECK_LAUNCH("fastdvd_output_grad");
    return SCI_OK;
}

extern "C" int sci_fastdvd_output_grad(const float* dout, float* dy, int B, int H, int W, int Cpad, void* stream) {
    return sci_fastdvd_output_grad_planes(dout, dy, B, 3, H, W, Cpad, stream);
}

extern "C" int sci_fastdvd_noisy_input(const float* v, const double* noise, float* vplus, long n, void* stream) {
    SCI_REQUIRE(v && noise && vplus && n > 0, "fastdvd_noisy_input");
    noisy_input_kernel<<<grid1d(n), 256, 0, sci_stream(stream)>>>(v, noise, vplus, n);
    SCI_CHECK_LAUNCH("fastdvd_noisy_input");
    return SCI_OK;
}

extern "C" int sci_meas_loss_fwd_bwd(const float* xhat, const float* phi, const float* y, float* dxhat, double* loss, int H,
                                     int W, int B, int C, long norm_pixels, void* stream) {
    SCI_REQUIRE(xhat && phi && y && loss && H > 0 && W > 0 && B > 0 && (C == 1 || C == 3) && norm_pixels >= 0, "meas_loss");
    // mean over `norm_pixels` (0 = this tensor's H*W; a row strip of a larger frame passes the frame's pixel count)
    const double cnt = norm_pixels > 0 ? (double)norm_pixels : (double)H * (double)W;
    meas_loss_kernel<<<grid1d((long)H * W), 256, 0, sci_stream(stream)>>>(xhat, phi, y, dxhat, loss, H, W, B, C,
                                                                          (float)(2.0 / cnt), 1.0 / cnt);
    SCI_CHECK_LAUNCH("meas_loss");
    return SCI_OK;
}

__global__ void axpy_kernel(const float* __restrict__ x, float a, const float* __restrict__ y, float* __restrict__ out, long n) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = x[i] + a * y[i];
}

extern "C" int sci_axpy(const float* x, float a, const float* y, float* out, long n, void* stream) {
    SCI_REQUIRE(x && y && out && n > 0, "axpy");
    axpy_kernel<<<(int)((n + 255) / 256), 256, 0, sci_stream(stream)>>>(x, a, y, out, n);
    SCI_CHECK_LAUNCH("axpy");
    return SCI_OK;
}

extern "C" int sci_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long n, double lr,
                             double beta1, double beta2, double eps, int step, void* stream) {
    SCI_REQUIRE(param && grad && exp_avg && exp_avg_sq && n > 0 && step >= 1, "adam_step");
    // python-double scalars as in torch.optim.adam._single_tensor_adam
    const double bc1 = 1.0 - pow(beta1, step), bc2 = 1.0 - pow(beta2, step);
    const float step_size = (float)(lr / bc1);
    const float bc2_sqrt = (float)sqrt(bc2);
    adam_kernel<<<grid1d(n), 256, 0, sci_stream(stream)>>>(param, grad, exp_avg, exp_avg_sq, n, (float)(1.0 - beta1),
                                                          (float)beta2, (float)(1.0 - beta2), (float)eps, step_size, bc2_sqrt);
    SCI_CHECK_LAUNCH("adam_step");
    return SCI_OK;
}
