// Boundary kernels of the DDnet deep demosaicker (models/network_demosaicking.py:377-463, packages/DDnet/DDnet_test.py:166-204).
//
// DDnet sees, for every centre frame f of the circular sequence, the five mosaics f-2..f+2 and evaluates
//   path 1: temp1 on the three 1-channel triples (full resolution),
//   path 2: temp11 on the three 4-channel (RGGB planes, half resolution) triples, + residual, bilinear x2, "fusion" convs,
//   temp2 on the three results of each path, and mixes the two temp2 outputs with learnable scalars.
// The conv stacks run on the tensor-core kernels (NHWC, 32-channel padded); the kernels here build their inputs from the
// frame-planar mosaics, apply the learnable input scalars, the residual adds, the up-sampling and the final mix.
// All HBM-bound index/elementwise work; compiled with --fmad=false (separate ATen ops in the reference).
//
// Batch order of the stacked triples: n = j*B + f  (j = 0,1,2 the triple, f the centre frame); triple j, slot k reads
// frame (f - 2 + j + k) mod B and the scalar a[3j+k]  (network_demosaicking.py:442-448).
//
// The forward kernels evaluate a range of centre frames [f0, f0+Bc) of the B-frame sequence (frame chunks that bound the
// memory of a pass): batch n = j*Bc + (f-f0), while the frame reads stay (f-2+j+k) mod B over the whole sequence.  The
// up-sampler also takes the global row of its local row 0 and the global frame height, so that it runs on a row strip of a
// larger frame (parallel.TileContext) with the source rows of the whole frame.  f0 = 0, Bc = B, row 0 = 0 is the whole.
#include "sci_common.cuh"

namespace {

__device__ __forceinline__ float rna_tf32(float v) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
    return __uint_as_float(r);
}

constexpr int DD_PIX = 256;       // pixels per block
constexpr int DD_CP = 32;         // channels of every packed tensor written here
constexpr int DD_CS = DD_CP + 1;  // padded shared-memory row

__device__ __forceinline__ int wrap(int f, int B) { return ((f % B) + B) % B; }

// channel k <- v (tf32 hi in k, remainder in k+16 when split)
__device__ __forceinline__ void put(float* row, int k, float v, int split) {
    if (split) {
        const float hi = rna_tf32(v);
        row[k] = hi;
        row[16 + k] = rna_tf32(v - hi);
    } else {
        row[k] = v;
    }
}

// cooperative, coalesced write of the block's [npx][32] rows
__device__ __forceinline__ void flush_rows(const float* srow, float* dst, int npx) {
    __syncthreads();
    for (int i = threadIdx.x; i < npx * DD_CP; i += DD_PIX) dst[i] = srow[(i / DD_CP) * DD_CS + (i % DD_CP)];
}

// path 1 input: out[j*Bc+f-f0][p][k] = mosaic[(f-2+j+k) mod B][p] * a[3j+k],  k = 0..2
__global__ void __launch_bounds__(DD_PIX) dd_pack1_kernel(const float* __restrict__ mosaic, const float* __restrict__ a,
                                                           float* __restrict__ out, int B, int f0, int Bc, long plane,
                                                           int split) {
    __shared__ float srow[DD_PIX * DD_CS];
    const int n = blockIdx.y, j = n / Bc, f = f0 + n % Bc;
    const long p0 = (long)blockIdx.x * DD_PIX, p = p0 + threadIdx.x;
    float* row = srow + threadIdx.x * DD_CS;
    for (int k = 0; k < DD_CP; ++k) row[k] = 0.f;
    if (p < plane) {
#pragma unroll
        for (int k = 0; k < 3; ++k) put(row, k, mosaic[(long)wrap(f - 2 + j + k, B) * plane + p] * a[3 * j + k], split);
    }
    flush_rows(srow, out + ((long)n * plane + p0) * DD_CP, (int)min((long)DD_PIX, plane - p0));
}

// path 2 input (half resolution): out[j*Bc+f-f0][y][x][4k+ib] = mosaic[fr][2y+ib/2][2x+ib%2] * a2[(3j+k)*4+ib]
__global__ void __launch_bounds__(DD_PIX) dd_pack4_kernel(const float* __restrict__ mosaic, const float* __restrict__ a2,
                                                           float* __restrict__ out, int B, int f0, int Bc, int H, int W,
                                                           int split) {
    __shared__ float srow[DD_PIX * DD_CS];
    const int n = blockIdx.y, j = n / Bc, f = f0 + n % Bc;
    const int h2 = H >> 1, w2 = W >> 1;
    const long plane = (long)H * W, hplane = (long)h2 * w2;
    const long p0 = (long)blockIdx.x * DD_PIX, p = p0 + threadIdx.x;
    float* row = srow + threadIdx.x * DD_CS;
    for (int k = 0; k < DD_CP; ++k) row[k] = 0.f;
    if (p < hplane) {
        const int y = (int)(p / w2), x = (int)(p % w2);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const float* src = mosaic + (long)wrap(f - 2 + j + k, B) * plane;
            const float2 top = *reinterpret_cast<const float2*>(src + (long)(2 * y) * W + 2 * x);
            const float2 bot = *reinterpret_cast<const float2*>(src + (long)(2 * y + 1) * W + 2 * x);
            const float* s = a2 + (3 * j + k) * 4;
            put(row, 4 * k + 0, top.x * s[0], split);
            put(row, 4 * k + 1, top.y * s[1], split);
            put(row, 4 * k + 2, bot.x * s[2], split);
            put(row, 4 * k + 3, bot.y * s[3], split);
        }
    }
    flush_rows(srow, out + ((long)n * hplane + p0) * DD_CP, (int)min((long)DD_PIX, hplane - p0));
}

// temp2 input of one path.  For centre frame f = f0+i:  v[j][c] = (mosaic ? mosaic[(f-1+j) mod B][p]*a[3j+1] : 0)
// + xo[j*Bc+i][p][c] (residual `in1 + x`, network_demosaicking.py:242, the 1-channel in1 broadcasting over 3 channels);
// t2in[i][p][3j+c] = v[j][c];  res[i][c][p] = v[1][c]  (the `in1` of the temp2 call, kept in full fp32).
__global__ void __launch_bounds__(DD_PIX) dd_mid_kernel(const float* __restrict__ mosaic, const float* __restrict__ a,
                                                         const float* __restrict__ xo, int Cp, float* __restrict__ t2in,
                                                         float* __restrict__ res, int B, int f0, int Bc, long plane,
                                                         int split) {
    __shared__ float srow[DD_PIX * DD_CS];
    const int i = blockIdx.y, f = f0 + i;
    const long p0 = (long)blockIdx.x * DD_PIX, p = p0 + threadIdx.x;
    float* row = srow + threadIdx.x * DD_CS;
    for (int k = 0; k < DD_CP; ++k) row[k] = 0.f;
    if (p < plane) {
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const float in1 = mosaic ? mosaic[(long)wrap(f - 1 + j, B) * plane + p] * a[3 * j + 1] : 0.f;
            const float* y = xo + ((long)(j * Bc + i) * plane + p) * Cp;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float v = mosaic ? in1 + y[c] : y[c];
                put(row, 3 * j + c, v, split);
                if (j == 1) res[((long)i * 3 + c) * plane + p] = v;
            }
        }
    }
    flush_rows(srow, t2in + ((long)i * plane + p0) * DD_CP, (int)min((long)DD_PIX, plane - p0));
}

// path 2 after the U-shaped body: y4[n][ib] = in1 + xo4 at half resolution (in1 = centre slot of the packed input),
// then nn.UpsamplingBilinear2d(scale_factor=2) (align_corners=True), written as the 4-channel input of the fusion convs.
// The H rows held start at global row row0 (even) of a frame of Ht rows: the source coordinate is formed from the global
// row; source rows outside the held ones (only for output rows within one row of the strip's edges, whose values the
// caller discards with its halo) are clamped to the held rows.
__global__ void __launch_bounds__(DD_PIX) dd_up4_kernel(const float* __restrict__ mosaic, const float* __restrict__ a2,
                                                         const float* __restrict__ xo4, int Cp, float* __restrict__ out,
                                                         int B, int f0, int Bc, int H, int W, int row0, int Ht, float sy,
                                                         float sx, int split) {
    __shared__ float srow[DD_PIX * DD_CS];
    const int n = blockIdx.y, j = n / Bc, f = f0 + n % Bc;
    const int h2 = H >> 1, w2 = W >> 1, ht2 = Ht >> 1, hr0 = row0 >> 1;
    const long plane = (long)H * W, hplane = (long)h2 * w2;
    const long p0 = (long)blockIdx.x * DD_PIX, p = p0 + threadIdx.x;
    float* row = srow + threadIdx.x * DD_CS;
    for (int k = 0; k < DD_CP; ++k) row[k] = 0.f;
    if (p < plane) {
        const int Y = (int)(p / W), X = (int)(p % W);
        // ATen area_pixel_compute_source_index + guard_index_and_lambda (align_corners=True)
        const float ry = sy * (float)(row0 + Y), rx = sx * (float)X;
        const int gy0 = min((int)ry, ht2 - 1), x0 = min((int)rx, w2 - 1);
        const int gy1 = min(gy0 + 1, ht2 - 1), x1 = min(x0 + 1, w2 - 1);
        const float ly1 = fminf(fmaxf(ry - (float)gy0, 0.f), 1.f), lx1 = fminf(fmaxf(rx - (float)x0, 0.f), 1.f);
        const float ly0 = 1.f - ly1, lx0 = 1.f - lx1;
        const int y0 = min(max(gy0 - hr0, 0), h2 - 1), y1 = min(max(gy1 - hr0, 0), h2 - 1);
        const float* src = mosaic + (long)wrap(f - 1 + j, B) * plane;
        const float* s = a2 + (3 * j + 1) * 4;
        const float* xb = xo4 + (long)n * hplane * Cp;
#pragma unroll
        for (int ib = 0; ib < 4; ++ib) {
            const int dy = ib >> 1, dx = ib & 1;
            auto val = [&](int yy, int xx) {
                return src[(long)(2 * yy + dy) * W + 2 * xx + dx] * s[ib] + xb[((long)yy * w2 + xx) * Cp + ib];
            };
            const float r0 = lx0 * val(y0, x0) + lx1 * val(y0, x1);
            const float r1 = lx0 * val(y1, x0) + lx1 * val(y1, x1);
            put(row, ib, ly0 * r0 + ly1 * r1, split);
        }
    }
    flush_rows(srow, out + ((long)n * plane + p0) * DD_CP, (int)min((long)DD_PIX, plane - p0));
}

// out[f][c][p] = a3[c]*(res1 + xo2[f][p][c]) + a3[3+c]*(res2 + xo2[B+f][p][c])      (:452-462)
__global__ void dd_final_kernel(const float* __restrict__ res1, const float* __restrict__ res2, const float* __restrict__ xo2,
                                int Cp, const float* __restrict__ a3, float* __restrict__ out, int B, long plane) {
    const long total = (long)B * 3 * plane;
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const long p = idx % plane;
    const int c = (int)((idx / plane) % 3), f = (int)(idx / (3 * plane));
    const float o1 = res1[idx] + __ldg(xo2 + ((long)f * plane + p) * Cp + c);
    const float o2 = res2[idx] + __ldg(xo2 + ((long)(B + f) * plane + p) * Cp + c);
    out[idx] = a3[c] * o1 + a3[3 + c] * o2;
}

// mosaic[f][p] = (rgb[f][0][p] + rgb[f][1][p]) + rgb[f][2][p]      (torch.sum(x, dim=1), :411-416)
__global__ void rgb_sum_kernel(const float* __restrict__ rgb, float* __restrict__ mosaic, int B, long plane) {
    const long total = (long)B * plane;
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const long p = idx % plane, f = idx / plane;
    const float* s = rgb + f * 3 * plane + p;
    mosaic[idx] = (s[0] + s[plane]) + s[2 * plane];
}

// =====================================================================================================
// Backward (self-supervised demosaicker update, DDnet_test.py:231-276): adjoints of the boundary kernels above.
// Gradients of the learnable scalars are block-reduced and added with atomics (the slots are zeroed by the caller).
// =====================================================================================================
__device__ __forceinline__ float block_sum_f(float v, float* scratch) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) scratch[wid] = v;
    __syncthreads();
    float r = 0.f;
    if (wid == 0) {
        r = lane < (int)((blockDim.x + 31) >> 5) ? scratch[lane] : 0.f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
    }
    return r;      // valid in thread 0
}

// loss = mean over [B][3][H][W] of (v - site(out))^2 with site(out) = out at the pixel's CFA channel, 0 elsewhere
// (DDnet_test.py:208-216, :268); dout = d loss / d out = (2/N) (site(out) - v) at the sites, 0 elsewhere.
__global__ void __launch_bounds__(256) dd_loss_kernel(const float* __restrict__ v, const float* __restrict__ out,
                                                       float* __restrict__ dout, double* __restrict__ loss, int B, int H, int W,
                                                       float norm, double inv_count) {
    __shared__ double red[32];
    const long plane = (long)H * W, total = (long)B * 3 * plane;
    const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    double err = 0.0;
    if (idx < total) {
        const long p = idx % plane;
        const int c = (int)((idx / plane) % 3);
        const int row = (int)(p / W), col = (int)(p % W);
        const bool site = c == (row & 1) + (col & 1);
        const float x = site ? out[idx] : 0.f;
        const float d = v[idx] - x;
        err = (double)(d * d);
        if (dout) dout[idx] = site ? norm * (x - v[idx]) : 0.f;
    }
    const double sblk = block_sum(err, red);
    if (threadIdx.x == 0) atomicAdd(loss, sblk * inv_count);
}

// out = a3[c]*o1 + a3[3+c]*o2, o_i = res_i + xo2[iB+f]:  d_xo2[iB+f][p][c] = a3[3i+c]*dout, d_res_i = the same (planar),
// da3[3i+c] += sum dout*o_i.  One thread per pixel, NHWC rows through shared memory.
__global__ void __launch_bounds__(DD_PIX) dd_final_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ res1,
                                                               const float* __restrict__ res2, const float* __restrict__ xo2,
                                                               int Cp, const float* __restrict__ a3, float* __restrict__ d_xo2,
                                                               float* __restrict__ d_res1, float* __restrict__ d_res2,
                                                               float* __restrict__ da3, int B, long plane) {
    __shared__ float srow[DD_PIX * DD_CS];
    __shared__ float red[32];
    const int f = blockIdx.y % B, i = blockIdx.y / B;        // i = 0: path 1, i = 1: path 2
    const long p0 = (long)blockIdx.x * DD_PIX, p = p0 + threadIdx.x;
    float* row = srow + threadIdx.x * DD_CS;
    for (int k = 0; k < DD_CP; ++k) row[k] = 0.f;
    float part[3] = {0.f, 0.f, 0.f};
    if (p < plane) {
        const float* res = i ? res2 : res1;
        float* dres = i ? d_res2 : d_res1;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const long o = ((long)f * 3 + c) * plane + p;
            const float g = dout[o];
            const float oi = res[o] + __ldg(xo2 + ((long)(i * B + f) * plane + p) * Cp + c);
            part[c] = g * oi;
            const float d = a3[3 * i + c] * g;
            row[c] = d;
            dres[o] = d;
        }
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float sblk = block_sum_f(part[c], red);
        if (threadIdx.x == 0) atomicAdd(da3 + 3 * i + c, sblk);
    }
    flush_rows(srow, d_xo2 + ((long)(i * B + f) * plane + p0) * DD_CP, (int)min((long)DD_PIX, plane - p0));
}

// adjoint of dd_mid_kernel: dv[j][c] = d_t2in[f][p][3j+c] + (j == 1 ? d_res[f][c][p] : 0);  d_xo[jB+f][p][c] = dv[j][c];
// path 1 (mosaic != NULL): da[3j+1] += sum_c dv[j][c] * mosaic[(f-1+j) mod B][p]
__global__ void __launch_bounds__(DD_PIX) dd_mid_bwd_kernel(const float* __restrict__ d_t2in, const float* __restrict__ d_res,
                                                             const float* __restrict__ mosaic, float* __restrict__ d_xo,
                                                             float* __restrict__ da, int B, long plane) {
    __shared__ float srow[DD_PIX * DD_CS];
    __shared__ float red[32];
    const int f = blockIdx.y % B, j = blockIdx.y / B;
    const long p0 = (long)blockIdx.x * DD_PIX, p = p0 + threadIdx.x;
    float* row = srow + threadIdx.x * DD_CS;
    for (int k = 0; k < DD_CP; ++k) row[k] = 0.f;
    float part = 0.f;
    if (p < plane) {
        const float* g = d_t2in + ((long)f * plane + p) * DD_CP + 3 * j;
        float s = 0.f;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            float dv = g[c];
            if (j == 1) dv += d_res[((long)f * 3 + c) * plane + p];
            row[c] = dv;
            s += dv;
        }
        if (mosaic) part = s * mosaic[(long)wrap(f - 1 + j, B) * plane + p];
    }
    if (mosaic) {
        const float sblk = block_sum_f(part, red);
        if (threadIdx.x == 0) atomicAdd(da + 3 * j + 1, sblk);
    }
    flush_rows(srow, d_xo + ((long)(j * B + f) * plane + p0) * DD_CP, (int)min((long)DD_PIX, plane - p0));
}

// da[3j+k] += sum_{f,p} d_in1[jB+f][p][k] * mosaic[(f-2+j+k) mod B][p]
__global__ void __launch_bounds__(256) dd_pack1_bwd_kernel(const float* __restrict__ d_in1, const float* __restrict__ mosaic,
                                                            float* __restrict__ da, int B, long plane) {
    __shared__ float red[32];
    const int n = blockIdx.y, j = n / B, f = n % B;
    const long p = (long)blockIdx.x * blockDim.x + threadIdx.x;
    float part[3] = {0.f, 0.f, 0.f};
    if (p < plane) {
        const float* g = d_in1 + ((long)n * plane + p) * DD_CP;
#pragma unroll
        for (int k = 0; k < 3; ++k) part[k] = g[k] * mosaic[(long)wrap(f - 2 + j + k, B) * plane + p];
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float sblk = block_sum_f(part[k], red);
        if (threadIdx.x == 0) atomicAdd(da + 3 * j + k, sblk);
    }
}

// path 2 scalars: da2[(3j+k)*4+ib] += sum d4[jB+f][y][x][ch] * mosaic[fr][2y+ib/2][2x+ib%2]
//   centre_only = 0: d4 is the gradient of the packed input, ch = 4k+ib, fr = f-2+j+k, all k
//   centre_only = 1: d4 is the gradient of y4 = in1 + xo4 (channels ib), i.e. of the centre slot k = 1 only
__global__ void __launch_bounds__(256) dd_pack4_bwd_kernel(const float* __restrict__ d4, const float* __restrict__ mosaic,
                                                            float* __restrict__ da2, int B, int H, int W, int centre_only) {
    __shared__ float red[32];
    const int n = blockIdx.y, j = n / B, f = n % B;
    const int h2 = H >> 1, w2 = W >> 1;
    const long plane = (long)H * W, hplane = (long)h2 * w2;
    const long p = (long)blockIdx.x * blockDim.x + threadIdx.x;
    const int y = (int)(p / w2), x = (int)(p % w2);
    for (int k = centre_only ? 1 : 0; k < (centre_only ? 2 : 3); ++k) {
        float part[4] = {0.f, 0.f, 0.f, 0.f};
        if (p < hplane) {
            const float* src = mosaic + (long)wrap(f - 2 + j + k, B) * plane;
            const float* g = d4 + ((long)n * hplane + p) * DD_CP + (centre_only ? 0 : 4 * k);
#pragma unroll
            for (int ib = 0; ib < 4; ++ib) part[ib] = g[ib] * src[(long)(2 * y + (ib >> 1)) * W + 2 * x + (ib & 1)];
        }
#pragma unroll
        for (int ib = 0; ib < 4; ++ib) {
            const float sblk = block_sum_f(part[ib], red);
            if (threadIdx.x == 0) atomicAdd(da2 + (3 * j + k) * 4 + ib, sblk);
        }
    }
}

// adjoint of the bilinear x2 (align_corners) up-sampling: scatter every full-resolution gradient to its four sources
__global__ void __launch_bounds__(256) dd_up4_bwd_kernel(const float* __restrict__ d_up, float* __restrict__ d_y4, int H, int W,
                                                          float sy, float sx) {
    const int n = blockIdx.y;
    const int h2 = H >> 1, w2 = W >> 1;
    const long plane = (long)H * W, hplane = (long)h2 * w2;
    const long p = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= plane) return;
    const int Y = (int)(p / W), X = (int)(p % W);
    const float ry = sy * (float)Y, rx = sx * (float)X;
    const int y0 = min((int)ry, h2 - 1), x0 = min((int)rx, w2 - 1);
    const int y1 = min(y0 + 1, h2 - 1), x1 = min(x0 + 1, w2 - 1);
    const float ly1 = fminf(fmaxf(ry - (float)y0, 0.f), 1.f), lx1 = fminf(fmaxf(rx - (float)x0, 0.f), 1.f);
    const float ly0 = 1.f - ly1, lx0 = 1.f - lx1;
    const float4 g = *reinterpret_cast<const float4*>(d_up + ((long)n * plane + p) * DD_CP);
    const float gv[4] = {g.x, g.y, g.z, g.w};
    float* base = d_y4 + (long)n * hplane * DD_CP;
#pragma unroll
    for (int ib = 0; ib < 4; ++ib) {
        atomicAdd(base + ((long)y0 * w2 + x0) * DD_CP + ib, ly0 * lx0 * gv[ib]);
        atomicAdd(base + ((long)y0 * w2 + x1) * DD_CP + ib, ly0 * lx1 * gv[ib]);
        atomicAdd(base + ((long)y1 * w2 + x0) * DD_CP + ib, ly1 * lx0 * gv[ib]);
        atomicAdd(base + ((long)y1 * w2 + x1) * DD_CP + ib, ly1 * lx1 * gv[ib]);
    }
}

inline int grid1d(long n, int block = 256) { return (int)((n + block - 1) / block); }

}  // namespace

#define DD_FRAMES_OK (B > 0 && f0 >= 0 && Bc > 0 && f0 + Bc <= B)

extern "C" int sci_ddnet_pack_input1_frames(const float* mosaic, const float* a, float* out, int B, int f0, int Bc, int H,
                                            int W, int Cpad, int split_tf32, void* stream) {
    SCI_REQUIRE(mosaic && a && out && DD_FRAMES_OK && H > 0 && W > 0 && Cpad == DD_CP, "ddnet_pack_input1");
    const long plane = (long)H * W;
    dd_pack1_kernel<<<dim3(grid1d(plane, DD_PIX), 3 * Bc), DD_PIX, 0, sci_stream(stream)>>>(mosaic, a, out, B, f0, Bc, plane,
                                                                                            split_tf32);
    SCI_CHECK_LAUNCH("ddnet_pack_input1");
    return SCI_OK;
}

extern "C" int sci_ddnet_pack_input1(const float* mosaic, const float* a, float* out, int B, int H, int W, int Cpad,
                                     int split_tf32, void* stream) {
    return sci_ddnet_pack_input1_frames(mosaic, a, out, B, 0, B, H, W, Cpad, split_tf32, stream);
}

extern "C" int sci_ddnet_pack_input4_frames(const float* mosaic, const float* a2, float* out, int B, int f0, int Bc, int H,
                                            int W, int Cpad, int split_tf32, void* stream) {
    SCI_REQUIRE(mosaic && a2 && out && DD_FRAMES_OK && H > 0 && W > 0 && H % 2 == 0 && W % 2 == 0 && Cpad == DD_CP,
                "ddnet_pack_input4");
    const long hplane = (long)(H / 2) * (W / 2);
    dd_pack4_kernel<<<dim3(grid1d(hplane, DD_PIX), 3 * Bc), DD_PIX, 0, sci_stream(stream)>>>(mosaic, a2, out, B, f0, Bc, H, W,
                                                                                             split_tf32);
    SCI_CHECK_LAUNCH("ddnet_pack_input4");
    return SCI_OK;
}

extern "C" int sci_ddnet_pack_input4(const float* mosaic, const float* a2, float* out, int B, int H, int W, int Cpad,
                                     int split_tf32, void* stream) {
    return sci_ddnet_pack_input4_frames(mosaic, a2, out, B, 0, B, H, W, Cpad, split_tf32, stream);
}

extern "C" int sci_ddnet_stage2_input_frames(const float* mosaic, const float* a, const float* xo, int xo_cpad, float* t2in,
                                             float* res, int B, int f0, int Bc, int H, int W, int Cpad, int split_tf32,
                                             void* stream) {
    SCI_REQUIRE(xo && t2in && res && DD_FRAMES_OK && H > 0 && W > 0 && Cpad == DD_CP && xo_cpad >= 3, "ddnet_stage2_input");
    SCI_REQUIRE((mosaic == nullptr) == (a == nullptr), "ddnet_stage2_input: mosaic and a go together");
    const long plane = (long)H * W;
    dd_mid_kernel<<<dim3(grid1d(plane, DD_PIX), Bc), DD_PIX, 0, sci_stream(stream)>>>(mosaic, a, xo, xo_cpad, t2in, res, B, f0,
                                                                                      Bc, plane, split_tf32);
    SCI_CHECK_LAUNCH("ddnet_stage2_input");
    return SCI_OK;
}

extern "C" int sci_ddnet_stage2_input(const float* mosaic, const float* a, const float* xo, int xo_cpad, float* t2in,
                                      float* res, int B, int H, int W, int Cpad, int split_tf32, void* stream) {
    return sci_ddnet_stage2_input_frames(mosaic, a, xo, xo_cpad, t2in, res, B, 0, B, H, W, Cpad, split_tf32, stream);
}

extern "C" int sci_ddnet_upsample4_strip(const float* mosaic, const float* a2, const float* xo4, int xo_cpad, float* out,
                                         int B, int f0, int Bc, int H, int W, int row0, int H_total, int Cpad, int split_tf32,
                                         void* stream) {
    SCI_REQUIRE(mosaic && a2 && xo4 && out && DD_FRAMES_OK && H >= 2 && W >= 4 && H % 2 == 0 && W % 2 == 0 &&
                Cpad == DD_CP && xo_cpad >= 4, "ddnet_upsample4");
    SCI_REQUIRE(row0 >= 0 && row0 % 2 == 0 && H_total >= 4 && H_total % 2 == 0 && row0 + H <= H_total,
                "ddnet_upsample4: rows [row0, row0+H) must be an even-aligned part of the H_total-row frame");
    const long plane = (long)H * W;
    // the scale factors of the WHOLE frame, with the float operations of ATen's area_pixel_compute_scale
    const float sy = (float)(H_total / 2 - 1) / (float)(H_total - 1), sx = (float)(W / 2 - 1) / (float)(W - 1);
    dd_up4_kernel<<<dim3(grid1d(plane, DD_PIX), 3 * Bc), DD_PIX, 0, sci_stream(stream)>>>(mosaic, a2, xo4, xo_cpad, out, B, f0,
                                                                                          Bc, H, W, row0, H_total, sy, sx,
                                                                                          split_tf32);
    SCI_CHECK_LAUNCH("ddnet_upsample4");
    return SCI_OK;
}

extern "C" int sci_ddnet_upsample4(const float* mosaic, const float* a2, const float* xo4, int xo_cpad, float* out, int B,
                                   int H, int W, int Cpad, int split_tf32, void* stream) {
    return sci_ddnet_upsample4_strip(mosaic, a2, xo4, xo_cpad, out, B, 0, B, H, W, 0, H, Cpad, split_tf32, stream);
}

extern "C" int sci_ddnet_output(const float* res1, const float* res2, const float* xo2, int xo_cpad, const float* a3,
                                float* out, int B, int H, int W, void* stream) {
    SCI_REQUIRE(res1 && res2 && xo2 && a3 && out && B > 0 && H > 0 && W > 0 && xo_cpad >= 3, "ddnet_output");
    const long plane = (long)H * W;
    dd_final_kernel<<<grid1d((long)B * 3 * plane), 256, 0, sci_stream(stream)>>>(res1, res2, xo2, xo_cpad, a3, out, B, plane);
    SCI_CHECK_LAUNCH("ddnet_output");
    return SCI_OK;
}

extern "C" int sci_rgb_sum(const float* rgb, float* mosaic, int H, int W, int B, void* stream) {
    SCI_REQUIRE(rgb && mosaic && B > 0 && H > 0 && W > 0, "rgb_sum");
    const long plane = (long)H * W;
    rgb_sum_kernel<<<grid1d((long)B * plane), 256, 0, sci_stream(stream)>>>(rgb, mosaic, B, plane);
    SCI_CHECK_LAUNCH("rgb_sum");
    return SCI_OK;
}

/* ---- backward entry points ---------------------------------------------------------------------------------- */
extern "C" int sci_ddnet_loss_fwd_bwd(const float* v, const float* out, float* dout, double* loss, int B, int H, int W,
                                      void* stream) {
    SCI_REQUIRE(v && out && loss && B > 0 && H > 0 && W > 0, "ddnet_loss_fwd_bwd");
    const long total = (long)B * 3 * H * W;
    dd_loss_kernel<<<grid1d(total), 256, 0, sci_stream(stream)>>>(v, out, dout, loss, B, H, W, 2.0f / (float)total, 1.0 / (double)total);
    SCI_CHECK_LAUNCH("ddnet_loss_fwd_bwd");
    return SCI_OK;
}

extern "C" int sci_ddnet_output_bwd(const float* dout, const float* res1, const float* res2, const float* xo2, int xo_cpad,
                                    const float* a3, float* d_xo2, float* d_res1, float* d_res2, float* da3, int B, int H, int W,
                                    void* stream) {
    SCI_REQUIRE(dout && res1 && res2 && xo2 && a3 && d_xo2 && d_res1 && d_res2 && da3 && B > 0 && H > 0 && W > 0 && xo_cpad >= 3,
                "ddnet_output_bwd");
    const long plane = (long)H * W;
    dd_final_bwd_kernel<<<dim3(grid1d(plane, DD_PIX), 2 * B), DD_PIX, 0, sci_stream(stream)>>>(dout, res1, res2, xo2, xo_cpad, a3,
                                                                                               d_xo2, d_res1, d_res2, da3, B, plane);
    SCI_CHECK_LAUNCH("ddnet_output_bwd");
    return SCI_OK;
}

extern "C" int sci_ddnet_stage2_input_bwd(const float* d_t2in, const float* d_res, const float* mosaic, float* d_xo, float* da,
                                          int B, int H, int W, void* stream) {
    SCI_REQUIRE(d_t2in && d_res && d_xo && B > 0 && H > 0 && W > 0, "ddnet_stage2_input_bwd");
    SCI_REQUIRE((mosaic == nullptr) == (da == nullptr), "ddnet_stage2_input_bwd: mosaic and da go together");
    const long plane = (long)H * W;
    dd_mid_bwd_kernel<<<dim3(grid1d(plane, DD_PIX), 3 * B), DD_PIX, 0, sci_stream(stream)>>>(d_t2in, d_res, mosaic, d_xo, da, B, plane);
    SCI_CHECK_LAUNCH("ddnet_stage2_input_bwd");
    return SCI_OK;
}

extern "C" int sci_ddnet_pack_input1_bwd(const float* d_in1, const float* mosaic, float* da, int B, int H, int W, void* stream) {
    SCI_REQUIRE(d_in1 && mosaic && da && B > 0 && H > 0 && W > 0, "ddnet_pack_input1_bwd");
    const long plane = (long)H * W;
    dd_pack1_bwd_kernel<<<dim3(grid1d(plane), 3 * B), 256, 0, sci_stream(stream)>>>(d_in1, mosaic, da, B, plane);
    SCI_CHECK_LAUNCH("ddnet_pack_input1_bwd");
    return SCI_OK;
}

extern "C" int sci_ddnet_pack_input4_bwd(const float* d4, const float* mosaic, float* da2, int B, int H, int W, int centre_only,
                                         void* stream) {
    SCI_REQUIRE(d4 && mosaic && da2 && B > 0 && H > 0 && W > 0 && H % 2 == 0 && W % 2 == 0, "ddnet_pack_input4_bwd");
    const long hplane = (long)(H / 2) * (W / 2);
    dd_pack4_bwd_kernel<<<dim3(grid1d(hplane), 3 * B), 256, 0, sci_stream(stream)>>>(d4, mosaic, da2, B, H, W, centre_only);
    SCI_CHECK_LAUNCH("ddnet_pack_input4_bwd");
    return SCI_OK;
}

extern "C" int sci_ddnet_upsample4_bwd(const float* d_up, float* d_y4, int B, int H, int W, void* stream) {
    SCI_REQUIRE(d_up && d_y4 && B > 0 && H >= 4 && W >= 4 && H % 2 == 0 && W % 2 == 0, "ddnet_upsample4_bwd");
    const long plane = (long)H * W;
    const float sy = (float)(H / 2 - 1) / (float)(H - 1), sx = (float)(W / 2 - 1) / (float)(W - 1);
    dd_up4_bwd_kernel<<<dim3(grid1d(plane), 3 * B), 256, 0, sci_stream(stream)>>>(d_up, d_y4, H, W, sy, sx);
    SCI_CHECK_LAUNCH("ddnet_upsample4_bwd");
    return SCI_OK;
}
