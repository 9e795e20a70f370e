// K4: Chambolle total-variation prior, fused with clip + ADMM dual update.
//
// Replaces the per-iteration  D2H -> skimage.restoration.denoise_tv_chambolle ->
// H2D  round trip of the reference (dvp_linear_inv_2_stage_ADMM_tensor_online.py
// :153-160, :403-407) plus the clip / dual update (:265-267, :501-503).
//
// Algorithm (SURVEY.md App. B, restated in oracle/tv_chambolle.py): each of the
// 4B channels (frame t, Bayer phase) is an independent (H/2)x(W/2) image that
// lives at stride 2 inside the full-resolution plane t.  n_iter_max = 5 means at
// most 4 dual updates shape the result, so the value at a pixel depends on a
// 4-pixel (half-res) neighbourhood: one block loads a full-res tile plus an
// 8-pixel halo into shared memory and runs ALL inner iterations there (halo
// recompute, no grid sync).  The early stop needs the per-channel energies
// E_0..E_3, which are global sums: the main pass assumes "no early stop" (true
// for ~97% of channel calls), writes deterministic per-block fp64 partial sums,
// a one-block decision kernel derives n_stop per channel, and a fix-up pass
// (same kernel, exits at once unless one of its four channels stopped early)
// rewrites the few channels that did.  No host involvement, 3 launches.
//
// Compiled with --fmad=false: the fp32 arithmetic mirrors numpy's separate ops.
#include "sci_common.cuh"

namespace {

constexpr int TV_TW = 64, TV_TH = 32;      // output tile (full-res pixels)
constexpr int TV_HALO = 8;                 // 4 half-res pixels
constexpr int TV_RW = TV_TW + 2 * TV_HALO; // 80
constexpr int TV_RH = TV_TH + 2 * TV_HALO; // 48
constexpr int TV_THREADS = 320;            // 40 column pairs x 8 row groups
constexpr int TV_MAX_UPD = 4;              // out_1..out_4 are the candidate results

// workspace: double epart[B][4 iters][2 kinds][4 phases][nblk], then int nstop[B*4]
__host__ __device__ inline size_t tv_epart_count(int B, int nblk) { return (size_t)B * 4 * 2 * 4 * nblk; }

// ---------------------------------------------------------------------------------------------------
// The tile kernel.  ncu on an earlier, straightforward form (one thread per column, profiles/ncu_r1_prof_tv_chambolle.csv)
// found it instruction-bound: issue slots 65 % busy, DRAM 2 %, and most instructions were boundary predicates and address
// arithmetic.  Hence
//   * the four shared-memory arrays carry a 2-pixel zero border, so tile-edge neighbours need no predicate (halo pixels
//     may then hold garbage one ring deeper per iteration, which the 8-pixel halo already budgets for);
//   * image borders are handled by per-row / per-thread select masks (dual variables outside the image stay exactly 0);
//   * a thread owns a PAIR of adjacent columns (the two column phases) of rows ry, ry+8, ..: every shared-memory access is
//     one 64-bit load/store for two pixels and the address arithmetic is shared.
// ---------------------------------------------------------------------------------------------------
constexpr int TV2_P = TV_RW + 4;                   // padded row pitch (84, even: float2 aligned)
constexpr int TV2_ROWS = TV_RH + 4;                // 52
constexpr int TV2_N = TV2_P * TV2_ROWS;            // 4368 floats per array
constexpr int TV2_PAIRS = TV_RW / 2;               // 40 column pairs
constexpr int TV2_RG = TV_THREADS / TV2_PAIRS;     // 8 row groups
constexpr int TV2_RPT = TV_RH / TV2_RG;            // 6 rows per thread

// Row-strip form (sci_tv_strip_*): the launch covers local rows [0, rows) of an H_total-row image whose first row is the
// global row row0 (even).  Border masks use global rows; the 8 rows above / below the strip are read from halo buffers
// [B][TV_HALO][W] that already hold f = x + c_b*b (null at a true image border, where the rows are zero as in the
// un-tiled kernel).  Rows further out than the halo may feed only pixels of the halo itself, never an own row.
struct TvStrip {
    int row0, H_total;
    const float* halo_top;
    const float* halo_bot;
    const unsigned* flag_top;     // peer-to-peer flag words to wait for before the halo is read (null: nothing to wait for)
    const unsigned* flag_bot;
    unsigned seq;
    unsigned* err;
};

// is_fix = 0: main pass (all channels run to n_iter_max, energies recorded)
// is_fix = 1: fix-up pass (only channels with nstop < last are rewritten)
// STRIP = false: the whole image, H rows (the TvStrip argument is unused).  STRIP = true: H is the strip's row count.
template <bool STRIP>
__global__ void __launch_bounds__(TV_THREADS, 3) tv_chambolle2_kernel(
    const float* __restrict__ x, const float* __restrict__ b, float c_b, float* __restrict__ theta,
    float* __restrict__ b_out, float s_b, int clip, int H, int W, float tau, float tw, int last_iter,
    double* __restrict__ epart, const int* __restrict__ nstop, int is_fix, TvStrip strip) {
    extern __shared__ float smem[];
    float* sf = smem;
    float* so = sf + TV2_N;
    float* sp0 = so + TV2_N;
    float* sp1 = sp0 + TV2_N;
    __shared__ int s_stop[4];

    const int t = blockIdx.z;
    const int nblk = gridDim.x * gridDim.y, blk = blockIdx.y * gridDim.x + blockIdx.x;
    if (threadIdx.x < 4) s_stop[threadIdx.x] = is_fix ? nstop[t * 4 + threadIdx.x] : last_iter;
    if (STRIP && threadIdx.x == 0) {
        // halo rows delivered peer to peer: a tile that reads them waits for the neighbour's sequence number (bounded, as in
        // halo_assemble_kernel: a lost neighbour sets the error word instead of hanging the GPU)
        const unsigned long long t0 = globaltimer_ns();
#pragma unroll
        for (int side = 0; side < 2; ++side) {
            const unsigned* flag = side == 0 ? (blockIdx.y == 0 ? strip.flag_top : nullptr)
                                             : ((int)blockIdx.y * TV_TH + TV_TH + TV_HALO > H ? strip.flag_bot : nullptr);
            if (!flag) continue;
            while ((int)(ld_acquire_sys(flag) - strip.seq) < 0) {
                if (globaltimer_ns() - t0 > 10000000000ull) { atomicExch(strip.err, 1u + side); break; }
                __nanosleep(200);
            }
        }
    }
    __syncthreads();
    if (is_fix && s_stop[0] >= last_iter && s_stop[1] >= last_iter && s_stop[2] >= last_iter && s_stop[3] >= last_iter)
        return;

    const int Himg = STRIP ? strip.H_total : H;                   // image height, for the border masks
    const int goff = STRIP ? strip.row0 : 0;                      // global row of local row 0
    const long plane = (long)H * W;
    const float* xp = x + t * plane;
    const float* bp = b ? b + t * plane : nullptr;
    const int gr0 = goff + blockIdx.y * TV_TH - TV_HALO, gc0 = blockIdx.x * TV_TW - TV_HALO;    // both even

    // zero everything once (borders stay zero for the whole kernel)
    {
        float4* z = reinterpret_cast<float4*>(smem);
        for (int i = threadIdx.x; i < 4 * TV2_N / 4; i += TV_THREADS) z[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    __syncthreads();

    const int cx = (threadIdx.x % TV2_PAIRS) * 2, ry = threadIdx.x / TV2_PAIRS;
    const int gc = gc0 + cx;                                  // even; the pair is (gc, gc+1) = column phases 0, 1
    const bool col_in = gc >= 0 && gc < W;                    // W even: both columns in or both out
    const bool col_right = col_in && gc + 2 < W;              // forward neighbour (c+2) exists in the image, for both
    const bool col_interior = cx >= TV_HALO && cx < TV_HALO + TV_TW && gc < W;
    const int rpar = ry & 1;                                  // gr0 even, rows advance by 8: fixed row parity per thread
    const int base = (ry + 2) * TV2_P + cx + 2;               // smem index of (rr = ry, cx)

    // ---- load f = x + c_b*b
#pragma unroll
    for (int k = 0; k < TV2_RPT; ++k) {
        const int gr = gr0 + ry + k * TV2_RG, lr = gr - goff, i = base + k * TV2_RG * TV2_P;
        float2 v = make_float2(0.f, 0.f);
        if (col_in && gr >= 0 && gr < Himg) {
            if (!STRIP || (lr >= 0 && lr < H)) {
                v = *reinterpret_cast<const float2*>(xp + (long)lr * W + gc);
                if (bp) {
                    const float2 bb = *reinterpret_cast<const float2*>(bp + (long)lr * W + gc);
                    v.x = v.x + c_b * bb.x; v.y = v.y + c_b * bb.y;
                }
            } else if (lr < 0) {
                v = *reinterpret_cast<const float2*>(strip.halo_top + ((long)t * TV_HALO + lr + TV_HALO) * W + gc);
            } else if (lr < H + TV_HALO) {
                v = *reinterpret_cast<const float2*>(strip.halo_bot + ((long)t * TV_HALO + lr - H) * W + gc);
            }
        }
        *reinterpret_cast<float2*>(sf + i) = v;
        *reinterpret_cast<float2*>(so + i) = v;
    }
    __syncthreads();

    double e_d[TV_MAX_UPD][2], e_n[TV_MAX_UPD][2];            // [iteration][column phase]
#pragma unroll
    for (int k = 0; k < TV_MAX_UPD; ++k) { e_d[k][0] = e_d[k][1] = e_n[k][0] = e_n[k][1] = 0.0; }
    const int stop0 = s_stop[rpar * 2 + 0], stop1 = s_stop[rpar * 2 + 1];

#pragma unroll
    for (int it = 0; it <= TV_MAX_UPD; ++it) {
        if (it > last_iter) break;
        if (it > 0) {
            // ---- phase A: d = -div p, out = f + d; write the result of the channels stopping here
#pragma unroll 2
            for (int k = 0; k < TV2_RPT; ++k) {
                const int rr = ry + k * TV2_RG, lr = gr0 - goff + rr, i = base + k * TV2_RG * TV2_P;
                const float2 p0 = *reinterpret_cast<const float2*>(sp0 + i), p1 = *reinterpret_cast<const float2*>(sp1 + i);
                const float2 pu = *reinterpret_cast<const float2*>(sp0 + i - 2 * TV2_P);
                const float2 pl = *reinterpret_cast<const float2*>(sp1 + i - 2);
                const float2 f = *reinterpret_cast<const float2*>(sf + i);
                float dx = -(p0.x + p1.x), dy = -(p0.y + p1.y);
                dx += pu.x; dy += pu.y;
                dx += pl.x; dy += pl.y;
                const float ox = f.x + dx, oy = f.y + dy;
                *reinterpret_cast<float2*>(so + i) = make_float2(ox, oy);
                if (col_interior && rr >= TV_HALO && rr < TV_HALO + TV_TH && lr < H) {     // own rows only
                    if (it < TV_MAX_UPD && !is_fix) {
                        e_d[it][0] += (double)(dx * dx);
                        e_d[it][1] += (double)(dy * dy);
                    }
                    const long g = (long)lr * W + gc;
                    const bool w0 = it == stop0 && (!is_fix || stop0 < last_iter);
                    const bool w1 = it == stop1 && (!is_fix || stop1 < last_iter);
                    if (w0 || w1) {
                        float t0 = ox, t1 = oy;
                        if (clip) { t0 = fminf(fmaxf(t0, 0.f), 1.f); t1 = fminf(fmaxf(t1, 0.f), 1.f); }
                        if (w0 && w1) {
                            *reinterpret_cast<float2*>(theta + t * plane + g) = make_float2(t0, t1);
                            if (bp) {
                                const float2 bb = *reinterpret_cast<const float2*>(bp + g), xx = *reinterpret_cast<const float2*>(xp + g);
                                *reinterpret_cast<float2*>(b_out + t * plane + g) =
                                    make_float2(bb.x + s_b * (xx.x - t0), bb.y + s_b * (xx.y - t1));
                            }
                        } else {
                            const int j = w0 ? 0 : 1;
                            const float th = w0 ? t0 : t1;
                            theta[t * plane + g + j] = th;
                            if (bp) b_out[t * plane + g + j] = bp[g + j] + s_b * (xp[g + j] - th);
                        }
                    }
                }
            }
            __syncthreads();
        }
        if (it == TV_MAX_UPD || it == last_iter) break;       // the last dual update never shapes the result
        // ---- phase B: forward differences, energy, dual update
#pragma unroll 2
        for (int k = 0; k < TV2_RPT; ++k) {
            const int rr = ry + k * TV2_RG, gr = gr0 + rr, i = base + k * TV2_RG * TV2_P;
            const bool in_img = col_in && gr >= 0 && gr < Himg;
            const bool has_dn = in_img && gr + 2 < Himg, has_rt = in_img && col_right;
            const float2 o = *reinterpret_cast<const float2*>(so + i);
            const float2 od = *reinterpret_cast<const float2*>(so + i + 2 * TV2_P);
            const float2 orr = *reinterpret_cast<const float2*>(so + i + 2);
            const float g0x = has_dn ? od.x - o.x : 0.f, g0y = has_dn ? od.y - o.y : 0.f;
            const float g1x = has_rt ? orr.x - o.x : 0.f, g1y = has_rt ? orr.y - o.y : 0.f;
            const float nx = sqrtf(g0x * g0x + g1x * g1x), ny = sqrtf(g0y * g0y + g1y * g1y);
            if (col_interior && rr >= TV_HALO && rr < TV_HALO + TV_TH && gr - goff < H && !is_fix) {
                e_n[it][0] += (double)nx;
                e_n[it][1] += (double)ny;
            }
            const float ix = 1.0f / (nx * tw + 1.0f), iy = 1.0f / (ny * tw + 1.0f);
            const float2 p0 = *reinterpret_cast<const float2*>(sp0 + i), p1 = *reinterpret_cast<const float2*>(sp1 + i);
            *reinterpret_cast<float2*>(sp0 + i) = in_img ? make_float2((p0.x - tau * g0x) * ix, (p0.y - tau * g0y) * iy)
                                                         : make_float2(0.f, 0.f);
            *reinterpret_cast<float2*>(sp1 + i) = in_img ? make_float2((p1.x - tau * g1x) * ix, (p1.y - tau * g1y) * iy)
                                                         : make_float2(0.f, 0.f);
        }
        __syncthreads();
    }

    if (is_fix) return;
    // ---- deterministic per-block energy partials: every thread parks its 16 sums in shared memory (the image arrays
    //      are dead now), 32 threads add them up in a fixed order
    __syncthreads();
    double* sd = reinterpret_cast<double*>(smem);             // [TV_THREADS][16]
#pragma unroll
    for (int k = 0; k < TV_MAX_UPD; ++k) {
        sd[threadIdx.x * 16 + k * 4 + 0] = e_d[k][0];
        sd[threadIdx.x * 16 + k * 4 + 1] = e_d[k][1];
        sd[threadIdx.x * 16 + k * 4 + 2] = e_n[k][0];
        sd[threadIdx.x * 16 + k * 4 + 3] = e_n[k][1];
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        // thread -> (k, kind, row parity rp, column phase cp)
        const int cp = threadIdx.x & 1, rp = (threadIdx.x >> 1) & 1, kind = (threadIdx.x >> 2) & 1, k = threadIdx.x >> 3;
        double s = 0.0;
        for (int g = rp; g < TV2_RG; g += 2)                  // row groups with this row parity
            for (int c = 0; c < TV2_PAIRS; ++c) s += sd[(g * TV2_PAIRS + c) * 16 + k * 4 + kind * 2 + cp];
        epart[((((size_t)t * 4 + k) * 2 + kind) * 4 + (rp * 2 + cp)) * nblk + blk] = s;
    }
}

// Fixed-order (deterministic) reduction of one channel's per-block partials: strided per-thread sums, then a tree.  The
// channel's 8 sums (q = k*2 + kind) end in sm[0][0..7].
constexpr int TV_DEC_THREADS = 128;
__device__ __forceinline__ void tv_channel_sums(const double* __restrict__ epart, int nblk, int t, int phase,
                                                double (*sm)[8]) {
    double acc[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {        // q = k*2 + kind
        const double* p = epart + ((((size_t)t * 4 + (q >> 1)) * 2 + (q & 1)) * 4 + phase) * nblk;
        double s = 0.0;
        for (int j = threadIdx.x; j < nblk; j += TV_DEC_THREADS) s += p[j];
        acc[q] = s;
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) sm[threadIdx.x][q] = acc[q];
    __syncthreads();
    for (int off = TV_DEC_THREADS / 2; off > 0; off >>= 1) {
        if (threadIdx.x < off) {
#pragma unroll
            for (int q = 0; q < 8; ++q) sm[threadIdx.x][q] += sm[threadIdx.x + off][q];
        }
        __syncthreads();
    }
}

// The reference's stopping rule  |E_prev - E_i| < eps * E_init  (i >= 1) on a channel's 8 energy sums.
__device__ __forceinline__ int tv_stop_rule(const double* e, double weight, double eps, double n_pix, int last_iter) {
    double E_init = 0.0, E_prev = 0.0;
    int stop = last_iter;
    for (int k = 0; k < TV_MAX_UPD && k < last_iter; ++k) {
        double E = e[k * 2 + 0];
        E += weight * e[k * 2 + 1];
        E /= n_pix;
        if (k == 0) { E_init = E; E_prev = E; }
        else if (fabs(E_prev - E) < eps * E_init) { stop = k; break; }
        else E_prev = E;
    }
    return stop;
}

// One block per channel: the reduction of tv_channel_sums, then the stopping rule (kept written out: the un-tiled decision
// compiles exactly as before).
__global__ void __launch_bounds__(TV_DEC_THREADS) tv_decide_kernel(const double* __restrict__ epart, int nblk, double weight,
                                                                   double eps, double n_pix, int last_iter,
                                                                   int* __restrict__ nstop, int* __restrict__ nstop_out) {
    __shared__ double sm[TV_DEC_THREADS][8];
    const int ch = blockIdx.x, t = ch >> 2, phase = ch & 3;
    double acc[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {        // q = k*2 + kind
        const double* p = epart + ((((size_t)t * 4 + (q >> 1)) * 2 + (q & 1)) * 4 + phase) * nblk;
        double s = 0.0;
        for (int j = threadIdx.x; j < nblk; j += TV_DEC_THREADS) s += p[j];
        acc[q] = s;
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) sm[threadIdx.x][q] = acc[q];
    __syncthreads();
    for (int off = TV_DEC_THREADS / 2; off > 0; off >>= 1) {
        if (threadIdx.x < off) {
#pragma unroll
            for (int q = 0; q < 8; ++q) sm[threadIdx.x][q] += sm[threadIdx.x + off][q];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        double E_init = 0.0, E_prev = 0.0;
        int stop = last_iter;
        for (int k = 0; k < TV_MAX_UPD && k < last_iter; ++k) {
            double E = sm[0][k * 2 + 0];
            E += weight * sm[0][k * 2 + 1];
            E /= n_pix;
            if (k == 0) { E_init = E; E_prev = E; }
            else if (fabs(E_prev - E) < eps * E_init) { stop = k; break; }
            else E_prev = E;
        }
        nstop[ch] = stop;
        if (nstop_out) nstop_out[ch] = stop;
    }
}

// Local half of a strip's decision: the same reduction as tv_decide_kernel, written out as esum[4B][8] for the
// cross-rank gather.  With one strip these are the un-tiled sums, bit for bit.
__global__ void __launch_bounds__(TV_DEC_THREADS) tv_strip_sums_kernel(const double* __restrict__ epart, int nblk,
                                                                       double* __restrict__ esum) {
    __shared__ double sm[TV_DEC_THREADS][8];
    const int ch = blockIdx.x, t = ch >> 2, phase = ch & 3;
    tv_channel_sums(epart, nblk, t, phase, sm);
    if (threadIdx.x < 8) esum[ch * 8 + threadIdx.x] = sm[0][threadIdx.x];
}

// Finish half: esum_all[world][4B][8] summed in rank order (every rank gets the same bits, hence the same decision),
// then the stopping rule.  One thread per channel.
__global__ void __launch_bounds__(TV_DEC_THREADS) tv_strip_decide_kernel(const double* __restrict__ esum_all, int world,
                                                                         int nch, double weight, double eps, double n_pix,
                                                                         int last_iter, int* __restrict__ nstop,
                                                                         int* __restrict__ nstop_out) {
    const int ch = blockIdx.x * TV_DEC_THREADS + threadIdx.x;
    if (ch >= nch) return;
    double e[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) e[q] = esum_all[ch * 8 + q];
    for (int r = 1; r < world; ++r) {
#pragma unroll
        for (int q = 0; q < 8; ++q) e[q] += esum_all[((size_t)r * nch + ch) * 8 + q];
    }
    const int stop = tv_stop_rule(e, weight, eps, n_pix, last_iter);
    nstop[ch] = stop;
    if (nstop_out) nstop_out[ch] = stop;
}

}  // namespace

extern "C" size_t sci_tv_workspace_bytes(int H, int W, int B) {
    if (H <= 0 || W <= 0 || B <= 0) return 0;
    const int nblk = sci_ceil_div(W, TV_TW) * sci_ceil_div(H, TV_TH);
    return tv_epart_count(B, nblk) * sizeof(double) + (size_t)B * 4 * sizeof(int);
}

extern "C" int sci_tv_chambolle2d(const float* x, const float* b, float c_b, float* theta, float* b_out, float s_b,
                                  int clip, int H, int W, int B, float weight, float eps, int n_iter_max,
                                  void* workspace, size_t workspace_bytes, int* nstop_out, void* stream) {
    SCI_REQUIRE(x && theta && workspace, "tv: null pointer");
    SCI_REQUIRE((b == nullptr) == (b_out == nullptr), "tv: b and b_out go together");
    SCI_REQUIRE(b == nullptr || b != b_out, "tv: b_out must not alias b");
    SCI_REQUIRE(H >= 2 && W >= 2 && H % 2 == 0 && W % 2 == 0 && B > 0 && B <= 65535, "tv: shape");
    if (n_iter_max < 1 || n_iter_max > TV_MAX_UPD + 1)
        return sci_fail(SCI_EUNSUPPORTED, "tv: n_iter_max must be in 1..5 (the reference uses 5)");
    if (workspace_bytes < sci_tv_workspace_bytes(H, W, B)) return sci_fail(SCI_EWORKSPACE, "tv: workspace too small");
    cudaStream_t st = sci_stream(stream);
    const dim3 grid(sci_ceil_div(W, TV_TW), sci_ceil_div(H, TV_TH), B);
    const int nblk = grid.x * grid.y;
    double* epart = reinterpret_cast<double*>(workspace);
    int* nstop = reinterpret_cast<int*>(epart + tv_epart_count(B, nblk));
    const size_t smem = (size_t)4 * TV2_N * sizeof(float);
    const cudaError_t e = sci_smem_limit((const void*)tv_chambolle2_kernel<false>, (int)smem);
    if (e != cudaSuccess) return sci_fail(SCI_ELAUNCH, "tv: smem attribute", e);
    const int last_iter = n_iter_max - 1;              // index of the last iterate (4 for n_iter_max=5)
    const float tau = 0.25f;                            // 1/(2*ndim), ndim = 2
    const float tw = (float)(0.25 / (double)weight);    // python-double tau/weight, cast at the fp32 multiply
    if (last_iter == 0) {
        // n_iter_max = 1 returns the input unchanged
        return sci_fail(SCI_EUNSUPPORTED, "tv: n_iter_max = 1 is the identity; not routed through the kernel");
    }
    tv_chambolle2_kernel<false><<<grid, TV_THREADS, smem, st>>>(x, b, c_b, theta, b_out, s_b, clip, H, W, tau, tw, last_iter, epart, nullptr, 0,
                                                             TvStrip{});
    SCI_CHECK_LAUNCH("tv main pass");
    const int nch = B * 4;
    tv_decide_kernel<<<nch, TV_DEC_THREADS, 0, st>>>(epart, nblk, (double)weight, (double)eps,
                                                     (double)(H / 2) * (double)(W / 2), last_iter, nstop, nstop_out);
    SCI_CHECK_LAUNCH("tv decide");
    tv_chambolle2_kernel<false><<<grid, TV_THREADS, smem, st>>>(x, b, c_b, theta, b_out, s_b, clip, H, W, tau, tw, last_iter, epart, nstop, 1,
                                                             TvStrip{});
    SCI_CHECK_LAUNCH("tv fix-up pass");
    return SCI_OK;
}

// ---------------------------------------------------------------------------------------------------
// Row strips of one frame (one strip per GPU).  A pixel's result depends only on rows within +-TV_HALO, for all
// n_iter_max <= 5 inner iterations, so one exchange of TV_HALO rows of f per call suffices; the only global coupling is
// the early stop, whose energies are reduced locally (sci_tv_strip_main), gathered across ranks by the caller and
// summed in rank order (sci_tv_strip_finish).
// ---------------------------------------------------------------------------------------------------
extern "C" size_t sci_tv_strip_workspace_bytes(int rows, int W, int B) { return sci_tv_workspace_bytes(rows, W, B); }

namespace {

// Every check runs before any CUDA call.
int tv_strip_check(const float* x, const float* b, const float* theta, const float* b_out, int rows, int W, int B, int row0,
                   int H_total, const float* halo_top, const float* halo_bot, int n_iter_max, const void* ws, size_t ws_bytes) {
    SCI_REQUIRE(x && theta && ws, "tv_strip: null pointer");
    SCI_REQUIRE((b == nullptr) == (b_out == nullptr), "tv_strip: b and b_out go together");
    SCI_REQUIRE(b == nullptr || b != b_out, "tv_strip: b_out must not alias b");
    SCI_REQUIRE(W >= 2 && W % 2 == 0 && B > 0 && B <= 65535, "tv_strip: shape");
    SCI_REQUIRE(rows >= TV_HALO && rows % 2 == 0 && row0 >= 0 && row0 % 2 == 0 && row0 + rows <= H_total,
                "tv_strip: rows and row0 must be even, rows >= 8, and the strip must lie inside the image");
    SCI_REQUIRE((row0 > 0) == (halo_top != nullptr) && (row0 + rows < H_total) == (halo_bot != nullptr),
                "tv_strip: a halo buffer is given exactly when a neighbouring strip exists");
    if (n_iter_max < 2 || n_iter_max > TV_MAX_UPD + 1)
        return sci_fail(SCI_EUNSUPPORTED, "tv_strip: n_iter_max must be in 2..5 (the reference uses 5)");
    if (ws_bytes < sci_tv_strip_workspace_bytes(rows, W, B)) return sci_fail(SCI_EWORKSPACE, "tv_strip: workspace too small");
    return SCI_OK;
}

}  // namespace

extern "C" int sci_tv_strip_main(const float* x, const float* b, float c_b, float* theta, float* b_out, float s_b, int clip,
                                 int rows, int W, int B, int row0, int H_total, const float* halo_top, const float* halo_bot,
                                 const unsigned* flag_top, const unsigned* flag_bot, unsigned seq, unsigned* err, float weight,
                                 float eps, int n_iter_max, void* workspace, size_t workspace_bytes, double* esum_out,
                                 void* stream) {
    const int rc = tv_strip_check(x, b, theta, b_out, rows, W, B, row0, H_total, halo_top, halo_bot, n_iter_max, workspace,
                                  workspace_bytes);
    if (rc != SCI_OK) return rc;
    SCI_REQUIRE(esum_out, "tv_strip: null esum_out");
    SCI_REQUIRE((flag_top == nullptr || halo_top) && (flag_bot == nullptr || halo_bot) && (!(flag_top || flag_bot) || err),
                "tv_strip: a flag word needs its halo buffer and the error word");
    (void)eps;
    cudaStream_t st = sci_stream(stream);
    const dim3 grid(sci_ceil_div(W, TV_TW), sci_ceil_div(rows, TV_TH), B);
    const int nblk = grid.x * grid.y;
    double* epart = reinterpret_cast<double*>(workspace);
    const size_t smem = (size_t)4 * TV2_N * sizeof(float);
    const cudaError_t e = sci_smem_limit((const void*)tv_chambolle2_kernel<true>, (int)smem);
    if (e != cudaSuccess) return sci_fail(SCI_ELAUNCH, "tv_strip: smem attribute", e);
    const float tau = 0.25f;
    const float tw = (float)(0.25 / (double)weight);
    const TvStrip strip{row0, H_total, halo_top, halo_bot, flag_top, flag_bot, seq, err};
    tv_chambolle2_kernel<true><<<grid, TV_THREADS, smem, st>>>(x, b, c_b, theta, b_out, s_b, clip, rows, W, tau, tw, n_iter_max - 1, epart,
                                                    nullptr, 0, strip);
    SCI_CHECK_LAUNCH("tv_strip main pass");
    tv_strip_sums_kernel<<<B * 4, TV_DEC_THREADS, 0, st>>>(epart, nblk, esum_out);
    SCI_CHECK_LAUNCH("tv_strip sums");
    return SCI_OK;
}

extern "C" int sci_tv_strip_finish(const float* x, const float* b, float c_b, float* theta, float* b_out, float s_b, int clip,
                                   int rows, int W, int B, int row0, int H_total, const float* halo_top, const float* halo_bot,
                                   float weight, float eps, int n_iter_max, void* workspace, size_t workspace_bytes,
                                   const double* esum_all, int world, int* nstop_out, void* stream) {
    const int rc = tv_strip_check(x, b, theta, b_out, rows, W, B, row0, H_total, halo_top, halo_bot, n_iter_max, workspace,
                                  workspace_bytes);
    if (rc != SCI_OK) return rc;
    SCI_REQUIRE(esum_all && world >= 1, "tv_strip: esum_all / world");
    cudaStream_t st = sci_stream(stream);
    const dim3 grid(sci_ceil_div(W, TV_TW), sci_ceil_div(rows, TV_TH), B);
    const int nblk = grid.x * grid.y, nch = B * 4;
    double* epart = reinterpret_cast<double*>(workspace);
    int* nstop = reinterpret_cast<int*>(epart + tv_epart_count(B, nblk));
    const size_t smem = (size_t)4 * TV2_N * sizeof(float);
    const cudaError_t e = sci_smem_limit((const void*)tv_chambolle2_kernel<true>, (int)smem);
    if (e != cudaSuccess) return sci_fail(SCI_ELAUNCH, "tv_strip: smem attribute", e);
    const int last_iter = n_iter_max - 1;
    const float tau = 0.25f;
    const float tw = (float)(0.25 / (double)weight);
    tv_strip_decide_kernel<<<sci_ceil_div(nch, TV_DEC_THREADS), TV_DEC_THREADS, 0, st>>>(
        esum_all, world, nch, (double)weight, (double)eps, (double)(H_total / 2) * (double)(W / 2), last_iter, nstop, nstop_out);
    SCI_CHECK_LAUNCH("tv_strip decide");
    // The fix-up pass reads the halo buffers again, without waiting: the main pass (earlier in this stream) has seen the
    // flags.  A peer-to-peer slot of parity p is rewritten only at exchange seq + 2, which the neighbour can issue only
    // after it has received this rank's halo of exchange seq + 1; this rank sends that after this pass in stream order,
    // so the slot is not overwritten while this pass reads it (sci_p2p.cu header).
    const TvStrip strip{row0, H_total, halo_top, halo_bot, nullptr, nullptr, 0u, nullptr};
    tv_chambolle2_kernel<true><<<grid, TV_THREADS, smem, st>>>(x, b, c_b, theta, b_out, s_b, clip, rows, W, tau, tw, last_iter, epart, nstop,
                                                    1, strip);
    SCI_CHECK_LAUNCH("tv_strip fix-up pass");
    return SCI_OK;
}
