/*
 * sci_b200.h — C ABI of the B200-native AdaptivePnP_SCI hot path.
 *
 * The reference (xyvirtualgroup/AdaptivePnP_SCI) is pure Python/PyTorch and has
 * no FFI of its own; the boundary of the hot path is the set of Python call
 * signatures listed in SURVEY.md §8(b).  This header is the C-ABI a binding
 * (ctypes, see adaptivepnp_sci_b200/_lib.py and INTEGRATION.md) loads to replace
 * the ATen/cuDNN/skimage op sequences behind those signatures.  Every entry
 * point cites the reference code it replaces (paths relative to the reference).
 *
 * Conventions
 *   - plain pointers and sizes only; all pointers are DEVICE pointers unless
 *     the name ends in _host; tensors stay owned by the caller (PyTorch);
 *   - stream-ordered: work is enqueued on `stream` (a cudaStream_t passed as
 *     void*), nothing synchronises, nothing allocates; kernels that need
 *     scratch take a workspace pointer whose size comes from a *_workspace_bytes
 *     query;
 *   - return 0 on success, a negative SCI_E* code on failure (never throws);
 *   - re-entrant across streams/devices (no global mutable state except the
 *     per-device TMA driver entry point cache).
 *
 * Device layouts ("planar"): the reference keeps cubes pixel-major
 * ([H,W,B], [h,w,B,4], [H,W,3,B]).  On the device every cube is FRAME-PLANAR
 * fp32:  Bayer-domain cubes  [B][H][W]   (full-resolution mosaic; the four
 * RGGB phases of the reference's [h,w,B,4] cubes are the (row&1,col&1) classes),
 * RGB cubes [B][3][H][W], planes [H][W].  Because the sensing operators are
 * pixel-wise, the per-phase loops of the reference (for ib in range(4)) are one
 * pass over the full-resolution planes.  sci_pixlast_to_planar /
 * sci_planar_to_pixlast convert at the boundary (bit-exact index remaps).
 */
#ifndef SCI_B200_H
#define SCI_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SCI_OK              0
#define SCI_EINVAL         -1   /* bad argument (null pointer, odd size, ...) */
#define SCI_ELAUNCH        -2   /* CUDA launch / runtime error               */
#define SCI_EUNSUPPORTED   -3   /* shape not supported by this build         */
#define SCI_EWORKSPACE     -4   /* workspace too small                       */

/* ABI version (major*1000+minor). */
int sci_version(void);
/* Last CUDA error string recorded by a failing call on this thread. */
const char* sci_last_error(void);

/* ---- layout remaps (bit-exact) -------------------------------------------
 * Replaces the strided-copy loops at dvp_linear_inv_2_stage_ADMM_tensor_online.py:66-82,
 * :170-172, :275-277, :312-314 and utils/utils_image.py:130-171.
 * pixel-last  in[P][C][B]  <->  planar out[B][C][P]   (C=1: Bayer cube, C=3: RGB cube) */
int sci_pixlast_to_planar(const float* in, float* out, int P, int C, int B, void* stream);
int sci_planar_to_pixlast(const float* in, float* out, int P, int C, int B, void* stream);

/* ---- K0: Bayer split + Phi-sum + initialisation --------------------------
 * dvp...online.py:59-82 / :347-370.  phi_hwb [H][W][B] (reference layout) ->
 * phi [B][H][W]; phisum [H][W] = sum_t phi, zeros replaced by 1 (:73);
 * theta0 [B][H][W] = y*phi_t (At_, utilspy.py:35-44) or, when x0_hwb != NULL,
 * the warm start x0_hwb [H][W][B] transposed (:82). */
int sci_bayer_split_init(const float* y, const float* phi_hwb, const float* x0_hwb,
                         float* phi, float* phisum, float* theta0,
                         int H, int W, int B, void* stream);

/* ---- sensing operators on arbitrary-stride views -------------------------
 * utilspy.py:28-33 (A_) and :35-44 (At_); strides in ELEMENTS so the
 * reference's Bayer-phase views ([h,w,B] slices of [h,w,B,4]) are accepted. */
int sci_A(const float* x, long sxh, long sxw, long sxt,
          const float* phi, long sph, long spw, long spt,
          float* y, long syh, long syw, int h, int w, int B, void* stream);
int sci_At(const float* y, long syh, long syw,
           const float* phi, long sph, long spw, long spt,
           float* x, long sxh, long sxw, long sxt, int h, int w, int B, void* stream);

/* ---- K1/K2: fused Euclidean projection ------------------------------------
 * stage 1 (dvp...online.py:389-391):  v = theta + b ;
 *     x = v + lambda * phi * ((y - sum_t phi*v) / (phisum + gamma))
 * stage 2 (dvp...online.py:128-140):  p = theta - (1/rho) b ;
 *     x = p + phi * ((y - sum_t phi*p) / (alpha*rho + phisum))
 * All cubes planar [B][npix].  If orig != NULL also accumulates
 * sse[0] += sum (x - orig)^2 (fp32 terms, fp64 sum) for the per-iteration PSNR
 * of stage 1 (:507-512). */
int sci_project_stage1(const float* theta, const float* b, const float* phi, const float* y,
                       const float* phisum, float* x, long npix, int B, float lambda_, float gamma,
                       const float* orig, double* sse, void* stream);
int sci_project_stage2(const float* theta, const float* b, const float* phi, const float* y,
                       const float* phisum, float* x, long npix, int B, double alpha, double rho,
                       void* stream);   /* alpha, rho are Python doubles in the reference: (1/rou) and alpha*rou are formed
                                           in double and cast to fp32 at the tensor op (dvp...online.py:131-140) */

/* ---- K4: TV prior (Chambolle projection) + fused dual update --------------
 * Replaces the D2H -> skimage.restoration.denoise_tv_chambolle(weight, n_iter_max=5,
 * multichannel=True) -> H2D round trip at dvp...online.py:153-160 / :403-407 and
 * the clip + dual update at :265-267 / :501-503.
 * Each of the 4B channels (frame t, Bayer phase) is an independent 2-D image of
 * (H/2)x(W/2) pixels living at stride 2 inside plane t.
 *     f     = x + c_b * b            (b may be NULL: f = x)
 *     theta = TV(f), clipped to [0,1] if clip != 0
 *     b_out = b + s_b * (x - theta)  (skipped if b == NULL)
 * b_out must not alias b (the early-stop fix-up pass re-reads b).
 * nstop_out (optional, may be NULL): int[4B], the iteration 1..4 whose iterate
 * was returned for channel t*4+phase.  workspace: sci_tv_workspace_bytes(). */
size_t sci_tv_workspace_bytes(int H, int W, int B);
int sci_tv_chambolle2d(const float* x, const float* b, float c_b, float* theta, float* b_out,
                       float s_b, int clip, int H, int W, int B, float weight, float eps,
                       int n_iter_max, void* workspace, size_t workspace_bytes, int* nstop_out,
                       void* stream);
/* K4 on a row strip of one frame (one strip per GPU).  The strip holds rows [row0, row0 + rows) of an
 * H_total-row image (row0, rows even, rows >= 8); x, b, theta, b_out are [B][rows][W].  A pixel's
 * result depends only on rows within +-8, so the caller provides, once per call, 8 rows of
 * f = x + c_b*b from each neighbour: halo_top / halo_bot [B][8][W], NULL exactly when the strip
 * touches that image border (see sci_halo_send_tv).  Every own pixel is then computed from the same
 * inputs in the same order as by sci_tv_chambolle2d.  The early stop is global, so the decision is
 * split in two:
 *   sci_tv_strip_main:   main pass + this strip's energy sums, esum_out double[4B][8];
 *   (caller: gather the esums of all strips in strip order, esum_all double[world][4B][8])
 *   sci_tv_strip_finish: sums esum_all in strip order, applies the stopping rule, writes nstop_out
 *                        (optional) and rewrites the channels that stopped early.
 * With one strip the result, nstop included, equals sci_tv_chambolle2d bit for bit.  With several,
 * the energies are summed in a different order, so a stop decision can differ from the un-tiled one
 * only when |E_prev - E_k| - eps*E_init is within fp64 rounding of zero.
 * flag_top / flag_bot (optional): local flag words of the peer-to-peer exchange; tiles that read a halo
 * first wait (bounded, ~10 s, then *err != 0) until the flag has reached seq.  n_iter_max in 2..5.
 * The workspace (sci_tv_strip_workspace_bytes) must be the same for main and finish. */
size_t sci_tv_strip_workspace_bytes(int rows, int W, int B);
int sci_tv_strip_main(const float* x, const float* b, float c_b, float* theta, float* b_out, float s_b, int clip,
                      int rows, int W, int B, int row0, int H_total, const float* halo_top, const float* halo_bot,
                      const unsigned* flag_top, const unsigned* flag_bot, unsigned seq, unsigned* err, float weight,
                      float eps, int n_iter_max, void* workspace, size_t workspace_bytes, double* esum_out,
                      void* stream);
int sci_tv_strip_finish(const float* x, const float* b, float c_b, float* theta, float* b_out, float s_b, int clip,
                        int rows, int W, int B, int row0, int H_total, const float* halo_top, const float* halo_bot,
                        float weight, float eps, int n_iter_max, void* workspace, size_t workspace_bytes,
                        const double* esum_all, int world, int* nstop_out, void* stream);

/* ---- K6: Malvar-2004 demosaic + (-w/tau) ----------------------------------
 * packages/colour_demosaicing/bayer/demosaicing/malvar2004.py:169-246 applied to
 * every frame (dvp...online.py:186-191) of the mosaic  m = x + c_b*b  (b may be
 * NULL), followed by x_rgb_w = x_rgb - inv_tau*w (:198).  Outputs planar
 * x_rgb [B][3][H][W] and, if w != NULL, u [B][3][H][W]. */
int sci_malvar2004(const float* x, const float* b, float c_b, const float* w, float inv_tau,
                   float* x_rgb, float* u, int H, int W, int B, void* stream);

/* ---- K3/K5: Bayer sampling of the denoised RGB + dual updates --------------
 * dvp...online.py:206-209 (theta <- RGGB samples of xhat), :265 (clip), :267
 * (b += x - theta), :271 (w += x_rgb - xhat), :275-280 (PSNR of merged theta).
 * first_iter != 0 reproduces the k=0 aliasing of xall/theta_all (:87-89): x is
 * replaced by the unclipped samples, so b receives theta_unclipped - theta. */
int sci_dual_update_rgb(const float* xhat, const float* x_rgb, float* w, const float* x,
                        float* b, float* theta, int first_iter, int H, int W, int B,
                        const float* orig, double* sse, void* stream);
/* Stage-1 bookkeeping of the deep branches of admm_denoise_bayer_demosaic_pre (dvp...online.py:439-503, single dual
 * variable): theta = clip(RGGB samples of xhat), b -= x - theta, sse[0] += sum (x - orig)^2 (PSNR of x, :507-512).
 * first_iter != 0 reproduces the k = 0 aliasing of xall / theta_all (:375-377): x is overwritten with the unclipped samples. */
int sci_dual_update_stage1(const float* xhat, float* x, float* b, float* theta, int first_iter, int H, int W, int B,
                           const float* orig, double* sse, void* stream);

/* Right/bottom reflect padding (torch F.pad mode='reflect') of `planes` [H][W] planes to [Ho][Wo] and the matching crop:
 * the sequence drivers pad every frame to a multiple of 4 before the network and cut the result back
 * (packages/fastdvdnet/fastdvdnet.py:119-141, packages/DDnet/DDnet_test.py:180-196). */
int sci_reflect_pad2d(const float* in, float* out, long planes, int H, int W, int Ho, int Wo, void* stream);
/* Right/bottom replication padding (torch.nn.ReplicationPad2d) of [planes][H][W] to [planes][Ho][Wo]: the odd-size path of
 * KAIR-FFDNet (models/network_ffdnet.py:56-59, cropped again at :68 with sci_crop2d). */
int sci_replicate_pad2d(const float* in, float* out, long planes, int H, int W, int Ho, int Wo, void* stream);
int sci_crop2d(const float* in, float* out, long planes, int H, int W, int Hc, int Wc, void* stream);
/* Closed-form demosaic update of the `close_form_demosaic` branch (dvp_linear_inv_2_stage_ADMM_tensor_online.py:112-118,
 * 175-182, 224-230), all frames in one launch:
 *   x_rgb[c] = (rho*x3[c] + b3[c] + tau*xhat[c] + w[c]) / (rho*m[c] + tau), optionally clipped to [0,1] (:182, FFDNet branch);
 *   u[c] = x_rgb[c] - inv_tau*w[c] (:198).  x, b [B][H][W] Bayer-domain; xhat, w, x_rgb, u [B][3][H][W]; x3/b3/m are the
 *   sparse 3-channel forms (fourCh2ThreeCh, utils_image.py:162-171) and the RGGB mask. */
int sci_closed_form_demosaic(const float* x, const float* b, const float* xhat, const float* w, float rho, float tau,
                             float inv_tau, int clip, float* x_rgb, float* u, int H, int W, int B, void* stream);
/* ---- K5: RGB cube -> Bayer samples / sparse 3-channel mosaic --------------
 * sci_rgb_to_bayer: dvp...online.py:206-209, packages/fastdvdnet/utils.py:69-78
 *   rgb [B][3][H][W] -> mosaic [B][H][W].
 * sci_bayer_to_rgb_sparse: utils/utils_image.py:153-161 (oneCh2ThreeCh). */
int sci_rgb_to_bayer(const float* rgb, float* mosaic, int H, int W, int B, void* stream);
int sci_bayer_to_rgb_sparse(const float* mosaic, float* rgb, int H, int W, int B, void* stream);

/* Reference-layout Bayer stack [h][w][B][4] <-> mosaic [H][W][B]
 * (utils/utils_image.py:130-151 fourCh2OneCh / oneCh2FourCh; B=1 covers the 3-D form). */
int sci_bayer4_to_mosaic(const float* stack, float* mosaic, int h, int w, int B, void* stream);
int sci_mosaic_to_bayer4(const float* mosaic, float* stack, int h, int w, int B, void* stream);

/* ---- K11: PSNR accumulation -------------------------------------------------
 * dvp...online.py:279,320: sse_per_frame[t] += sum_p (a[t][p]-orig[t][p])^2,
 * fp32 difference and square, fp64 accumulation (skimage PSNR restated). */
int sci_psnr_accum(const float* a, const float* orig, long npix, int B, double* sse_per_frame,
                   void* stream);
/* Per-frame SSIM of the final report (dvp...online.py:321; skimage structural_similarity defaults: 7x7 uniform window,
 * sample covariance, K1 = .01, K2 = .03, float64, mean over the image cropped by 3 pixels), evaluated on the device:
 * ssim_sum[t] += sum of the SSIM map over the crop of frame t (divide by (H-6)*(W-6)).  a, ref [B][H][W]. */
int sci_ssim_accum(const float* a, const float* ref, int H, int W, int B, double data_range, double* ssim_sum,
                   void* stream);


/* =========================================================================
 * Denoiser networks: 3x3 convolutions as implicit GEMM (K7-K10)
 * Replaces the cuDNN/ATen conv stacks of models/network_ffdnet.py:54-69 and
 * packages/fastdvdnet/models.py:16-253 (forward) and the autograd graph built by
 * the online fine-tune adapters (test_ffdnet_ipol.py:248-299, test_fastdvdnet.py:343-451).
 *
 * Activations are NHWC fp32 with the channel count padded to a multiple of 32
 * (16 for pure outputs); padded channels hold zeros.  Weights are pre-packed by
 * sci_conv_pack_weights into [9 taps][Cout][Cin] (Cin contiguous = K-major).
 * impl: SCI_CONV_TC  = tcgen05/TMEM tensor-core kernel fed by TMA (TF32 operands, fp32 accumulate)
 *       SCI_CONV_REF = fp32 FFMA implicit-GEMM (on-device numerics reference)
 * ========================================================================= */
#define SCI_CONV_TC  0
#define SCI_CONV_REF 1

typedef struct sci_conv_desc {
    const float* x;         /* input  [N][H][W][Cin]                                              */
    const float* w;         /* packed weights [9][Cout][Cin]                                      */
    const float* scale;     /* per output column, NULL = 1   (folded BatchNorm gamma/sqrt(var+eps)) */
    const float* shift;     /* per output column, NULL = 0   (bias, or folded BatchNorm shift)      */
    const float* residual;  /* added after activation, same layout as y, NULL = none (skip add)    */
    float* y;               /* output [N][Ho][Wo][Cout], or [N][2Ho][2Wo][Cout/4] if pixel_shuffle  */
    int N, H, W;            /* input batch and spatial size                                        */
    int Cin, Cout;          /* padded channel counts (Cin % 8 == 0; TC: Cin % 32 == 0, Cout % 16 == 0) */
    int stride;             /* 1 or 2 (pad 1): Ho = (H-1)/stride+1                                  */
    int relu;               /* ReLU after scale/shift                                             */
    int pixel_shuffle;      /* 1: GEMM column q*(Cout/4)+c goes to sub-pixel q=(dy*2+dx), channel c */
    int round_tf32;         /* 1: round stored outputs to TF32 (they feed the next tensor-core conv) */
    int w_split;            /* TC only. 1: w is [18][Cout][Cin] = tf32(w) in taps 0..8 and the remainder
                               tf32(w - tf32(w)) in taps 9..17 (sci_conv_pack_weights round_tf32 = 2); both are
                               multiplied, which removes the weight-rounding error of the TF32 path.
                               With half_io: the fp16 SPLIT FORM of the FFDNet inference chain (stride 1, Cout <= 128) - x, w and y
                               carry, per group of 32 channels, a 64-channel chunk [32 fp16 values | their 32 remainders
                               (v - fp16(v)) * 2^11]: Cin = 64 * groups, Cout_store = 2 * Cout, w from
                               sci_conv_pack_weights_half(ci_dup = -1).  value x value goes to one accumulator, value x
                               remainder + remainder x value to a second one, added (x 2^-11) in the epilogue: the
                               accuracy of the "3xTF32" scheme at the fp16 tensor rate and half the bytes */
    int emit_lo;            /* TC only. 1: y has 2*Cout channels per pixel: [tf32(v) | tf32(v - tf32(v))]; the next
                               layer is packed with ci_dup = Cout so it multiplies both ("3xTF32": ~fp32 accuracy) */
    const float* planar_in1; /* TC only, with planar_out: [N][P][H][W] frames, P = planar_planes                */
    float* planar_out;      /* TC only. non-NULL: the layer is the last conv of a FastDVDnet DenBlock (Cout == 32, 3 real
                               channels): instead of y the kernel writes out[n][c][h][w] = planar_in1[n][c][h][w] - conv[c]
                               (packages/fastdvdnet/models.py:196) as planar frames; y may be NULL */
    int pdl;                /* TC only. 1: programmatic dependent launch — the kernel may be scheduled while the previous kernel
                               of the stream is still draining; it sets up barriers / TMEM / resident weights meanwhile and
                               waits for that kernel's completion before touching x / residual / planar_in1.  Only valid when
                               the previous kernel does not write w, scale or shift (engine: inference chains) */
    int half_io;            /* TC only. 1: x, w, residual and y hold IEEE binary16 values (the pointers are typed float* for the
                               ABI only); kind::f16 MMAs with fp32 accumulation - the same 11-bit significand as TF32 at half
                               the bytes and twice the tensor rate.  scale / shift / planar_in1 / planar_out stay fp32.  Cin is
                               then the K extent of the packed weights (a multiple of 64), Cout the GEMM columns (multiple of 32);
                               inference chains only (the weight-gradient kernels read fp32 activations) */
    int Cin_store;          /* half_io: channels per pixel of the stored input tensor (<= Cin, multiple of 8; the K columns
                               beyond it are zero-filled by TMA); 0 = Cin */
    int Cout_store;         /* half_io: channels per pixel of the stored output tensor (every pixel row written is 64 channels:
                               real columns, then zeros; rows sticking out of the tensor are clipped); 0 = Cout (Cout/4 with
                               pixel_shuffle) */
    const float* mask_y;    /* TC only (fp32, stride-1 kernel). non-NULL: this call is a DATA GRADIENT whose output is the gradient
                               w.r.t. the stored output `mask_y` (same layout as y) of the PRECEDING layer, and that layer's
                               activation backward is fused into the epilogue: y = (conv [+ residual]) * (mask_y > 0 if mask_relu),
                               col_s1[c] += sum y, col_s2[c] += sum y * mask_y over all pixels (either may be NULL; the sums the
                               bias / BatchNorm parameter gradients need, see sci_act_bwd / sci_bn_param_grad).  Replaces the
                               separate sci_act_bwd pass over dy, y and dz */
    float* col_s1;
    float* col_s2;
    int mask_relu;
    int lo_channel0;        /* TC only, with w_split on an input written with emit_lo: first channel of the remainder half
                               [tf32(v) | tf32(v - tf32(v))] (= the producing layer's Cout).  The small products then accumulate
                               in their own TMEM accumulator and are added in the epilogue (fewer truncating accumulations into
                               the main sum).  0 = one accumulator */
    int K_used;             /* TC only. > 0: only the first K_used input channels (K columns of the packed weights) can be non-zero;
                               the MMAs over the all-zero tail of the last 128-byte channel chunk are skipped (results unchanged).
                               0 = Cin */
    int planar_planes;      /* TC only, with planar_out: planes P per frame of planar_in1 / planar_out, 3 (colour) or 1 (the
                               gray FastDVDnet: columns 1 and 2 of the layer, all-zero weights in the colour-shaped embedding,
                               are not written).  0 = 3 */
    void* workspace;        /* with mask_y and col_s1: NULL = the column sums are added with atomics (their low bits depend on
                               the order in which CTAs finish); non-NULL = FIXED-ORDER column sums, bit-identical on every run:
                               each CTA stores its sums (epilogue warps added in warp order) into its own slot of this
                               workspace, and a second kernel of the same call adds the slots in slot order into col_s1 /
                               col_s2.  Size: sci_conv3x3_fwd_workspace_bytes (SCI_EINVAL when smaller).  16-byte aligned */
    size_t workspace_bytes;
} sci_conv_desc;

/* 1 if this build contains the tcgen05 tensor-core convolution kernels. */
int sci_conv_tc_available(void);
/* y = act(scale * conv3x3(x, w) + shift) [+ residual].  Forward pass of every layer; the data-gradient
 * of a stride-1 layer is the same call with weights packed in transposed+flipped form. */
int sci_conv3x3_fwd(const sci_conv_desc* d, int impl, void* stream);
int sci_conv3x3_dgrad(const sci_conv_desc* d, int impl, void* stream);
/* Bytes of sci_conv_desc.workspace the fixed-order column sums of this call need with this impl: 0 unless the call is a
 * fused data gradient (mask_y) with column sums (col_s1) on the tensor-core path.  Otherwise slots x 2 x C x 4, C = the
 * stored output channels (Cout, Cout/4 with pixel_shuffle), one slot [col_s1 part | col_s2 part] per CTA of each launch
 * (a 256-column layer runs as two launches of the same grid).  Host arithmetic only. */
size_t sci_conv3x3_fwd_workspace_bytes(const sci_conv_desc* d, int impl);

typedef struct sci_wgrad_desc {
    const float* x;         /* layer input  [N][H][W][Cin]                          */
    const float* dz;        /* grad wrt GEMM output [N][Ho][Wo][Cout]               */
    const float* oscale;    /* per output column scale (folded BN), NULL = 1        */
    float* dw;              /* packed weight gradient [9][Cout][Cin], ACCUMULATED   */
    int N, H, W, Cin, Cout, stride;
    void* workspace;        /* NULL = every CTA adds its partial gradient into dw with atomics (low bits depend on the order
                               in which CTAs finish); non-NULL = FIXED ORDER, bit-identical on every run: CTA column b stores
                               its scaled partial into slot b (a [9][Cout][Cin] block) of this workspace, and a second kernel
                               of the same call computes dw[i] = dw[i] + (((slot0[i] + slot1[i]) + slot2[i]) + ...).  Size:
                               sci_conv3x3_wgrad_workspace_bytes (SCI_EINVAL when smaller).  16-byte aligned */
    size_t workspace_bytes;
} sci_wgrad_desc;
/* dw[tap][co][ci] += oscale[co] * sum_{n,ho,wo} dz[n,ho,wo,co] * x[n, ho*s+r-1, wo*s+q-1, ci] */
int sci_conv3x3_wgrad(const sci_wgrad_desc* d, int impl, void* stream);
/* Bytes of sci_wgrad_desc.workspace for this impl: slots x 9 x Cout x Cin x 4, slots = the CTA columns of the launch (a
 * function of the shape only: tensor-core v3 min(tiles, 148), v2 min(tiles, 148 / (3 m_tiles)), fp32 reference its pixel
 * chunks).  0 for a descriptor the impl rejects.  Host arithmetic only. */
size_t sci_conv3x3_wgrad_workspace_bytes(const sci_wgrad_desc* d, int impl);

/* PyTorch weight [Co][Ci/groups][3][3] -> packed [9][Co_pad][Ci_pad] (zero padded; grouped convs become
 * block-diagonal; ps != 0 permutes output columns for PixelShuffle(2): column q*(Co/4)+c <- channel c*4+q).
 * transpose_flip != 0 packs the data-gradient form [9][Ci_pad][Co_pad] with taps flipped and rows scaled by
 * oscale (may be NULL).  round_tf32 = 1 rounds to TF32 (RNA); round_tf32 = 2 (forward form only) writes the split
 * form [18][Co_pad][Ci_pad]: tf32(w) in taps 0..8 and tf32(w - tf32(w)) in taps 9..17 (see sci_conv_desc.w_split).
 * ci_dup > 0 (first layers on the tensor-core path): input channels [ci_dup, ci_dup+Ci) get the SAME weights as
 * [0, Ci).  The network-boundary packers put tf32(v) in channel k and the remainder tf32(v - tf32(v)) in channel
 * k + ci_dup, so the first layer sees its input at ~2^-22 relative precision at no extra cost (K is padded to 32
 * anyway); sci_conv_unpack_wgrad then sums the two gradient blocks. */
int sci_conv_pack_weights(const float* w, float* packed, int Co, int Ci, int groups, int Co_pad, int Ci_pad,
                          int ps, const float* oscale, int transpose_flip, int round_tf32, int ci_dup, void* stream);
/* fp16 form of the forward packing for sci_conv_desc.half_io layers: packed [9][Co_pad][Ci_pad] IEEE binary16, round to
 * nearest; Ci_pad % 64 == 0 (one 128-byte operand row = 64 channels) or Ci_pad == 32 (64-byte rows).  Same grouped / PixelShuffle / ci_dup rules as above
 * (the fp16 network-boundary packer puts fp16(v) in channel k and fp16(v - fp16(v)) in channel k + ci_dup).
 * ci_dup = -1: split form (sci_conv_desc.w_split with half_io): Ci_pad = 64 * ceil(Ci / 32), K chunk g = [fp16(w) of channels
 * 32g..32g+31 | (w - fp16(w)) * 2^11 of the same channels]. */
int sci_conv_pack_weights_half(const float* w, void* packed, int Co, int Ci, int groups, int Co_pad, int Ci_pad, int ps,
                               int ci_dup, void* stream);
/* fp16 form of sci_fastdvd_pack_input (packages/fastdvdnet/models.py:185 input block, circular window fastdvdnet.py:115):
 * out [B][H][W][C] binary16 (C = 32 or 64), channels 0..11 = fp16 of [f0 RGB, sigma, f1 RGB, sigma, f2 RGB, sigma], 16..27 =
 * the fp16 remainders, others zero. */
int sci_fastdvd_pack_input_half(const float* frames, float sigma, void* out, int B, int H, int W, int C, void* stream);
/* The same with frames of NC planes (3, or 1 for gray frames: channels slot*4+1 and slot*4+2 are then +0, bit for bit what
 * packing the zero-embedded colour cube gives).  sci_fastdvd_pack_input_half is this with NC = 3. */
int sci_fastdvd_pack_input_half_planes(const float* frames, float sigma, void* out, int B, int NC, int H, int W, int C,
                                       void* stream);
/* Data-gradient weights of a STRIDE-2 layer (groups = 1) as a sub-pixel convolution over dz at the low resolution:
 * packed [9][4*Ci_pad][Co_pad]; run sci_conv3x3_dgrad with x = dz [N][Ho][Wo][Co_pad], Cin = Co_pad, Cout = 4*Ci_pad,
 * stride 1, pixel_shuffle = 1 -> dx [N][2Ho][2Wo][Ci_pad].  Replaces "zero-dilate dz, then convolve at full resolution"
 * (4x less operand traffic, no dilated tensor).  oscale (may be NULL) scales by the folded BatchNorm scale of column co. */
int sci_conv_pack_weights_s2t(const float* w, float* packed, int Co, int Ci, int Co_pad, int Ci_pad, const float* oscale,
                              int round_tf32, void* stream);
/* inverse of the forward packing for gradients: dw_torch[Co][Ci/groups][3][3] = packed_dw (assign) */
int sci_conv_unpack_wgrad(const float* packed_dw, float* dw, int Co, int Ci, int groups, int Co_pad, int Ci_pad,
                          int ps, int ci_dup, void* stream);

/* Batched per-layer bookkeeping: one launch runs a whole TABLE of the small operations above / below (device-resident array
 * of n_ops entries; blockIdx.y = entry, max_blocks = ceil(largest element count / 256)).  kind: 0 sci_conv_pack_weights
 * (a = w, b = oscale, o0 = packed; tflip / round_tf32 / ci_dup as there), 1 sci_conv_pack_weights_s2t, 2
 * sci_conv_pack_weights_half, 3 sci_conv_unpack_wgrad (a = packed_dw, o0 = dw), 4 sci_bn_fold (a gamma, b beta, c mean,
 * d var, eps -> o0 scale, o1 shift; C = Co, C_pad = Co_pad), 5 sci_bn_param_grad (a s1, b s2, c gamma, d beta -> o0 dgamma,
 * o1 dbeta), 6 copy of Co floats a -> o0.  Entries of one table must not depend on each other. */
typedef struct sci_layer_op {
    int kind;
    int Co, Ci, groups, Co_pad, Ci_pad, ps, tflip, round_tf32, ci_dup;
    float eps;
    const void *a, *b, *c, *d;
    void *o0, *o1;
} sci_layer_op;
int sci_layer_ops_batch(const sci_layer_op* table_device, int n_ops, int max_blocks, void* stream);

/* BatchNorm (eval mode, packages/fastdvdnet/models.py:21-26) folded to per-column scale/shift:
 * scale = gamma*rsqrt(var+eps), shift = beta - mean*scale; columns >= C are zeroed up to C_pad. */
int sci_bn_fold(const float* gamma, const float* beta, const float* mean, const float* var, float eps,
                float* scale, float* shift, int C, int C_pad, void* stream);
/* Backward of y = relu(scale*conv+shift):  dz = dy * (y > 0) (relu != 0) else dy, written to dz (may alias dy);
 * s1[c] += sum dz, s2[c] += sum dz*y  (either may be NULL).  n_pix pixels of C channels (NHWC). */
int sci_act_bwd(const float* dy, const float* y, float* dz, long n_pix, int C, int relu, float* s1, float* s2,
                void* stream);
/* The same with FIXED-ORDER column sums (bit-identical on every run; dz is the same as sci_act_bwd's): block b stores its
 * (s1, s2) partials into slot b = [C floats of s1 | C floats of s2] of the workspace, a second kernel adds the slots in slot
 * order into s1 / s2.  workspace: sci_act_bwd_workspace_bytes(n_pix, C) bytes, 16-byte aligned; missing or smaller ->
 * SCI_EINVAL before any launch. */
size_t sci_act_bwd_workspace_bytes(long n_pix, int C);
int sci_act_bwd_ordered(const float* dy, const float* y, float* dz, long n_pix, int C, int relu, float* s1, float* s2,
                        void* workspace, size_t workspace_bytes, void* stream);
/* BatchNorm affine gradients from the two sums: dbeta = s1, dgamma = (s2 - beta*s1)/gamma (0 where gamma == 0). */
int sci_bn_param_grad(const float* s1, const float* s2, const float* gamma, const float* beta, float* dgamma,
                      float* dbeta, int C, void* stream);

/* NHWC helpers for the backward pass: pixel-unshuffle of a gradient ([N][2H][2W][C] -> [N][H][W][4C], column
 * q*C+c) and zero-dilation by 2 ([N][H][W][C] -> [N][2H][2W][C]) for the data-gradient of stride-2 layers. */
int sci_nhwc_pixel_unshuffle(const float* in, float* out, int N, int H, int W, int C, void* stream);
int sci_nhwc_dilate2(const float* in, float* out, int N, int H, int W, int C, void* stream);

/* FFDNet boundary (models/network_ffdnet.py:56-68, models/basicblock.py:104-126); C = 3 (colour) or 1 (gray):
 * pack:   u [B][C][H][W] planar -> head input [B][H/2][W/2][Cpad]: channel c*4+dy*2+dx = u[c][2h+dy][2w+dx],
 *         channel 4C = sigma, rest 0 (round_tf32: tf32(v) in channel k and the remainder in channel k+16).
 * unpack: tail output [B][H/2][W/2][Cpad] (column c*4+dy*2+dx) -> xhat [B][3][H][W] planar (PixelShuffle(2)).
 * unpack_grad: d xhat planar -> d tail output (adjoint of unpack). */
int sci_ffdnet_pack_input(const float* u, float sigma, float* out, int B, int C, int H, int W, int Cpad, int round_tf32,
                          void* stream);
int sci_ffdnet_unpack_output(const float* y, float* xhat, int B, int C, int H, int W, int Cpad, void* stream);
int sci_ffdnet_unpack_output_grad(const float* dxhat, float* dy, int B, int C, int H, int W, int Cpad, void* stream);
/* fp16 split form of the same boundary (inference chain, sci_conv_desc.w_split + half_io): out [B][H/2][W/2][64] binary16 =
 * [fp16(v_k), k < 32 | fp16((v_k - fp16(v_k)) * 2^11)] with v as in sci_ffdnet_pack_input; unpack reads a tail of the same
 * form and writes xhat = value + remainder * 2^-11 as planar fp32. */
int sci_ffdnet_pack_input_split_half(const float* u, float sigma, void* out, int B, int C, int H, int W, void* stream);
int sci_ffdnet_unpack_output_split_half(const void* y, float* xhat, int B, int C, int H, int W, void* stream);

/* FastDVDnet boundary (packages/fastdvdnet/models.py:185,196,234; fastdvdnet.py:115 circular window):
 * pack:   frames [B][3][H][W] planar -> DenBlock input [B][H][W][Cpad], for block f the channels
 *         [F(f-1) rgb, sigma, F(f) rgb, sigma, F(f+1) rgb, sigma] with circular frame indices, rest 0.
 *         (temp1 is evaluated once per centre frame: the B distinct triples of the circular 5-window; temp2 of
 *         output frame f then reads the temp1 results f-1, f, f+1 through the same packer.)
 * output: out[f][c] = frames_center[f][c] - y[f][h][w][c]  (models.py:196), y = last conv [B][H][W][Cpad].
 * The two *_grad entry points are the adjoints used by the fine-tune backward pass. */
int sci_fastdvd_pack_input(const float* frames, float sigma, float* out, int B, int H, int W, int Cpad,
                           int round_tf32, void* stream);
int sci_fastdvd_output(const float* frames, const float* y, float* out, int B, int H, int W, int Cpad, void* stream);
int sci_fastdvd_output_grad(const float* dout, float* dy, int B, int H, int W, int Cpad, void* stream);
int sci_fastdvd_pack_input_grad(const float* din, float* dframes, int B, int H, int W, int Cpad, int accumulate,
                                void* stream);
/* The four above for frames of NC planes: 3 (the entry points above are these with NC = 3) or 1 (gray FastDVDnet in the
 * colour-shaped embedding: frames / out / dout / dframes [B][1][H][W]; the packer writes the frame into channel slot*4 and +0
 * into slot*4+1..2, the output kernels read or write column / plane 0 only).  For NC = 1 every result is bit for bit the NC = 3
 * result on the zero-embedded cube (plane 0 of it for the planar outputs). */
int sci_fastdvd_pack_input_planes(const float* frames, float sigma, float* out, int B, int NC, int H, int W, int Cpad,
                                  int round_tf32, void* stream);
int sci_fastdvd_output_planes(const float* frames, const float* y, float* out, int B, int NC, int H, int W, int Cpad,
                              void* stream);
int sci_fastdvd_output_grad_planes(const float* dout, float* dy, int B, int NC, int H, int W, int Cpad, void* stream);
int sci_fastdvd_pack_input_grad_planes(const float* din, float* dframes, int B, int NC, int H, int W, int Cpad, int accumulate,
                                       void* stream);
/* ---- DDnet deep-demosaic boundary (models/network_demosaicking.py:377-463; packages/DDnet/DDnet_test.py:166-204) ----
 * mosaic [B][H][W] planar (the sum over the three sparse colour planes DDnet takes, :411-416 — sci_rgb_sum).
 * The triples of the circular 5-window are stacked as batch n = j*B + f (j = triple 0..2, f = centre frame); triple j,
 * slot k reads frame (f-2+j+k) mod B scaled by the learnable scalar a[3j+k] (:398-399, :442-448).  Every packed tensor
 * is NHWC with Cpad == 32; split_tf32 != 0 stores tf32(v) in channel k and the remainder in channel k+16.
 *   pack_input1 : path 1 (temp1) input  [3B][H][W][32],   channels 0..2   = the three scaled mosaics
 *   pack_input4 : path 2 (temp11) input [3B][H/2][W/2][32], channel 4k+ib = RGGB plane ib of slot k, scaled by a2[3j+k][ib]
 *   stage2_input: xo [3B][H][W][xo_cpad] = last conv of a path; v[j][c] = in1 + xo (residual :242; in1 = mosaic*a[3j+1],
 *                 or 0 when mosaic == NULL: path 2, whose residual was applied before the up-sampling);
 *                 t2in[f][p][3j+c] = v[j][c] (temp2 input), res[f][c][p] = v[1][c] (temp2's own in1, full fp32)
 *   upsample4   : y4 = in1 + xo4 at half resolution, nn.UpsamplingBilinear2d(x2, align_corners=True) (:371) ->
 *                 [3B][H][W][32] input of the fusion convs
 *   output      : out[f][c] = a3[0][c]*(res1 + xo2[f]) + a3[1][c]*(res2 + xo2[B+f])   (:452-462), xo2 [2B][H][W][xo_cpad] */
int sci_rgb_sum(const float* rgb, float* mosaic, int H, int W, int B, void* stream);
int sci_ddnet_pack_input1(const float* mosaic, const float* a, float* out, int B, int H, int W, int Cpad, int split_tf32,
                          void* stream);
int sci_ddnet_pack_input4(const float* mosaic, const float* a2, float* out, int B, int H, int W, int Cpad, int split_tf32,
                          void* stream);
int sci_ddnet_stage2_input(const float* mosaic, const float* a, const float* xo, int xo_cpad, float* t2in, float* res,
                           int B, int H, int W, int Cpad, int split_tf32, void* stream);
int sci_ddnet_upsample4(const float* mosaic, const float* a2, const float* xo4, int xo_cpad, float* out, int B, int H,
                        int W, int Cpad, int split_tf32, void* stream);
int sci_ddnet_output(const float* res1, const float* res2, const float* xo2, int xo_cpad, const float* a3, float* out,
                     int B, int H, int W, void* stream);
/* Frame chunks and row strips of the same kernels.  *_frames evaluate the centre frames [f0, f0+Bc) of the B-frame
 * sequence (0 <= f0, Bc > 0, f0+Bc <= B): batch n = j*Bc + (f-f0) in out / xo / t2in / res (Bc frames), frame reads stay
 * (f-2+j+k) mod B over the whole mosaic [B][H][W].  upsample4_strip also takes the global row row0 (even) of the first of
 * the H rows held and the height H_total of the whole frame (row0 + H <= H_total): the bilinear source coordinate is that
 * of the whole frame, source rows outside the held ones are clamped to them (output rows within one row of a strip edge
 * whose neighbour rows are not held are therefore not those of the whole frame; a caller with a halo discards them).
 * The whole-frame entry points above are these with f0 = 0, Bc = B, row0 = 0, H_total = H. */
int sci_ddnet_pack_input1_frames(const float* mosaic, const float* a, float* out, int B, int f0, int Bc, int H, int W,
                                 int Cpad, int split_tf32, void* stream);
int sci_ddnet_pack_input4_frames(const float* mosaic, const float* a2, float* out, int B, int f0, int Bc, int H, int W,
                                 int Cpad, int split_tf32, void* stream);
int sci_ddnet_stage2_input_frames(const float* mosaic, const float* a, const float* xo, int xo_cpad, float* t2in,
                                  float* res, int B, int f0, int Bc, int H, int W, int Cpad, int split_tf32, void* stream);
int sci_ddnet_upsample4_strip(const float* mosaic, const float* a2, const float* xo4, int xo_cpad, float* out, int B,
                              int f0, int Bc, int H, int W, int row0, int H_total, int Cpad, int split_tf32, void* stream);
/* Backward of the DDnet boundary (self-supervised demosaicker update, DDnet_test.py:231-276).
 *   loss_fwd_bwd     : loss += mean over [B][3][H][W] of (v - site(out))^2, site() keeps the RGGB site of each channel
 *                      (DDnet_test.py:208-216, :268); dout (may be NULL) = d loss / d out
 *   output_bwd       : adjoint of sci_ddnet_output: d_xo2 [2B][H][W][32], d_res1/d_res2 [B][3][H][W], da3[6] += ...
 *   stage2_input_bwd : adjoint of sci_ddnet_stage2_input for one path: d_xo [3B][H][W][32]; path 1 also da[3j+1] += ...
 *   pack_input1_bwd  : da[3j+k] += <d_in1[jB+f][.][k], mosaic[(f-2+j+k) mod B]>
 *   pack_input4_bwd  : da2[(3j+k)*4+ib] += ...; centre_only = 1 treats d4 as the gradient of y4 = in1 + xo4 (slot k = 1)
 *   upsample4_bwd    : adjoint of the bilinear x2 up-sampling, scattered (atomics) into the ZEROED d_y4 [3B][H/2][W/2][32]
 * The scalar-gradient slots (da, da2, da3) are accumulated with atomics and must be zeroed by the caller. */
int sci_ddnet_loss_fwd_bwd(const float* v, const float* out, float* dout, double* loss, int B, int H, int W, void* stream);
int sci_ddnet_output_bwd(const float* dout, const float* res1, const float* res2, const float* xo2, int xo_cpad, const float* a3,
                         float* d_xo2, float* d_res1, float* d_res2, float* da3, int B, int H, int W, void* stream);
int sci_ddnet_stage2_input_bwd(const float* d_t2in, const float* d_res, const float* mosaic, float* d_xo, float* da, int B, int H,
                               int W, void* stream);
int sci_ddnet_pack_input1_bwd(const float* d_in1, const float* mosaic, float* da, int B, int H, int W, void* stream);
int sci_ddnet_pack_input4_bwd(const float* d4, const float* mosaic, float* da2, int B, int H, int W, int centre_only, void* stream);
int sci_ddnet_upsample4_bwd(const float* d_up, float* d_y4, int B, int H, int W, void* stream);
/* training input of the FastDVDnet fine-tune (test_fastdvdnet.py:359 with utils_image.py:183-192):
 * vplus = v + float32(float64(v) + noise), noise float64 from the host RNG. */
int sci_fastdvd_noisy_input(const float* v, const double* noise, float* vplus, long n, void* stream);

/* HOST function (no GPU work): numpy's LEGACY normal generator, bit for bit, multi-threaded.
 * out_host[n] = loc + scale * legacy_gauss() exactly as np.random.RandomState.normal(loc, scale, n) would produce from
 * the MT19937 state (key[624], pos, has_gauss, gauss), which is advanced in place.  Replaces the single-threaded draw
 * inside add_gaussian_noise_meas_cuda (utils/utils_image.py:183-192). */
int sci_host_legacy_normal(uint32_t* key_host, int* pos_host, int* has_gauss_host, double* gauss_host, double loc,
                           double scale, double* out_host, long n, int nthreads);

/* Measurement-consistency loss of the online fine-tune (test_ffdnet_ipol.py:275-291,
 * test_fastdvdnet.py:428-431):  m = RGGB samples of xhat; up = sum_t m_t*phi_t;
 * loss += mean((up - y)^2) over H*W (fp64 accumulate);  dxhat[t][c][p] = phi_t * 2(up-y)/(H*W) at the
 * Bayer colour of p, 0 elsewhere (C = 3; with C = 1 xhat is a gray cube [B][1][H][W] and m = xhat).  dxhat may be NULL (loss only).  norm_pixels = 0 normalises by this tensor's
 * H*W; a row strip of a spatially tiled frame passes the pixel count of the WHOLE frame. */
int sci_meas_loss_fwd_bwd(const float* xhat, const float* phi, const float* y, float* dxhat, double* loss,
                          int H, int W, int B, int C, long norm_pixels, void* stream);
/* Gray-scale stage-2 bookkeeping (derived FFDNet-gray configuration, no Bayer sampling): theta = clip(xhat);
 * b += x - theta (first_iter: x := xhat, the k=0 aliasing of dvp...online.py:87-89); w += x_pre - xhat; optional PSNR. */
int sci_dual_update_gray(const float* xhat, const float* x_pre, float* w, const float* x, float* b, float* theta,
                         int first_iter, long n, const float* orig, double* sse, void* stream);
/* out = x + a*y (the merged mosaic x + b/rho of a row strip before its halo rows are exchanged, SURVEY 8(e)). */
int sci_axpy(const float* x, float a, const float* y, float* out, long n, void* stream);

/* Adam step over a flat parameter bucket (torch.optim.Adam defaults: betas (0.9,0.999), eps 1e-8, no weight
 * decay; test_ffdnet_ipol.py:251, test_fastdvdnet.py:385).  step is 1-based. */
int sci_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long n, double lr,
                  double beta1, double beta2, double eps, int step, void* stream);

/* ---- peer-to-peer halo exchange (spatial row-strip tiling of one large frame, BASELINE config 5; SURVEY 8(b) export
 * `sci_halo_exchange`, 8(e) row 3).  Replaces the reference-side "one GPU holds the whole frame" with strips whose boundary
 * rows are stored straight into the neighbouring GPU's memory over NVLink.
 * sci_p2p_alloc / get_handle / open_handle: a cudaMalloc'ed, zeroed region, its 64-byte CUDA IPC handle, and the mapping
 * of a neighbour's region into this process (peer access enabled lazily).  The caller exchanges the handles once
 * (torch.distributed object all-gather).
 * sci_halo_send: copies the first / last `halo` rows of own [planes][rows][W] (fp32) into up_dst / down_dst (PEER pointers,
 * NULL = no neighbour on that side), then release-stores `seq` into up_flag / down_flag (peer flag words).
 * sci_halo_assemble (same stream): waits until *flag_top / *flag_bot (LOCAL flag words written by the neighbours) have
 * reached `seq`, then writes ext [planes][top + rows + bot][W] = [recv_top | own | recv_bot].  *err becomes non-zero if a
 * neighbour did not deliver within ~10 s (the wait is bounded: a lost peer must not hang the GPU).
 * sci_halo_send_tv: the TV prior's halo (sci_tv_strip_main).  Like sci_halo_send, but stores f = x + c_b*b of the
 * first / last `halo` rows of x, b [planes][rows][W] (b may be NULL: f = x; W even), rounded exactly as the TV kernel
 * forms it; the receiver reads its slots in place. */
int sci_p2p_alloc(size_t bytes, void** ptr);
int sci_p2p_free(void* ptr);
int sci_p2p_get_handle(void* ptr, void* handle64);
int sci_p2p_open_handle(const void* handle64, void** ptr);
int sci_p2p_close_handle(void* ptr);
int sci_halo_send(const float* own, int planes, int rows, int W, int halo, float* up_dst, float* down_dst,
                  unsigned* up_flag, unsigned* down_flag, unsigned seq, unsigned* done_counter, void* stream);
int sci_halo_send_tv(const float* x, const float* b, float c_b, int planes, int rows, int W, int halo, float* up_dst,
                     float* down_dst, unsigned* up_flag, unsigned* down_flag, unsigned seq, unsigned* done_counter,
                     void* stream);
int sci_halo_assemble(const float* own, int planes, int rows, int W, int top, int bot, const float* recv_top,
                      const float* recv_bot, const unsigned* flag_top, const unsigned* flag_bot, unsigned seq,
                      float* ext, unsigned* err, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SCI_B200_H */
