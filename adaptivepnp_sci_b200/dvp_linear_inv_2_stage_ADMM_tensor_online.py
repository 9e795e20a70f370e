"""The two ADMM solvers of AdaptivePnP_SCI, B200-native.

Drop-in for the reference module of the same name: ``admm_denoise_bayer_demosaic_pre``
(dvp_linear_inv_2_stage_ADMM_tensor_online.py:326-552, stage 1 / TV warm start) and
``twoStageAdmm_denoise_bayer`` (:40-324, stage 2 / plug-and-play deep denoiser with
online adaptation) keep the reference's names, argument order, defaults, array
layouts at the boundary, return tuples and ``ValueError`` for unknown denoisers.

What differs is everything between the boundary and the hardware:

* the solver state (theta, b, x, Phi, w, x_rgb) lives on the device in frame-planar
  layout for the whole reconstruction; the host sees scalars only (the reference
  copies the cube D2H every iteration for PSNR and D2H+H2D for TV);
* one fused kernel per ADMM step instead of ~40 ATen launches:
  ``sci_project_stage1/2`` (A, At, projection, optional PSNR),
  ``sci_tv_chambolle2d`` (TV prior + clip + dual update, early stop on device),
  ``sci_malvar2004`` (merge + demosaic of all frames + ``-w/tau``),
  ``sci_dual_update_rgb`` (Bayer sampling + clip + both dual updates + PSNR);
* the denoisers run through the native conv kernels (see ``ffdnet_adapter`` /
  ``fastdvdnet_adapter``).

There is no CPU or PyTorch-op fallback: without the CUDA library the import fails.
"""
import os
import sys

import numpy as np
import torch

from . import iqa, ops
from .utils_image import cuda2np, np2tch_cuda  # noqa: F401  (np2tch_cuda is imported from here by the scripts)

__all__ = ["admm_denoise_bayer_demosaic_pre", "twoStageAdmm_denoise_bayer", "twoStageAdmm_denoise_gray", "np2tch_cuda",
           "cuda2np"]


def _as_list(sigma, iter_max):
    if not isinstance(sigma, list):
        sigma = [sigma]
    if not isinstance(iter_max, list):
        iter_max = [iter_max] * len(sigma)
    return sigma, iter_max


def _to_device(a):
    if torch.is_tensor(a):
        return a.to(device="cuda", dtype=torch.float32).contiguous()
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()


class _Problem:
    """Device-resident problem data shared by both stages (K0)."""

    def __init__(self, y_bayer, Phi_bayer, x0_bayer, X_orig):
        y = _to_device(y_bayer)
        phi_hwb = _to_device(Phi_bayer)
        x0 = None if x0_bayer is None else _to_device(x0_bayer)
        self.H, self.W, self.B = phi_hwb.shape
        if self.H % 2 or self.W % 2:
            raise ValueError("Bayer measurements need even height and width, got %dx%d" % (self.H, self.W))
        self.y = y
        self.phi, self.phisum, self.theta = ops.bayer_split_init(y, phi_hwb, x0)
        self.x = torch.empty_like(self.theta)
        self.b = torch.zeros_like(self.theta)
        self.npix = self.H * self.W
        self.orig = None
        if X_orig is not None:
            self.orig = ops.pixlast_to_planar(_to_device(X_orig), 1, self.B).view(self.B, self.H, self.W)

    def to_hwb(self, cube):
        """planar [B,H,W] -> numpy [H,W,B] (the layout the reference returns)."""
        return cuda2np(ops.planar_to_pixlast(cube, 1, self.B).view(self.H, self.W, self.B))

    def frame_iqa(self, cube, x_np, X_orig):
        psnr_, ssim_ = [], []
        if X_orig is not None:
            sse = torch.zeros(self.B, dtype=torch.float64, device=cube.device)
            ops.psnr_accum(cube, self.orig, sse)
            ss = ops.ssim_frames(cube, self.orig)                    # on-device SSIM (skimage defaults, fp64), :321
            p = iqa.psnr_from_sse(sse.cpu().numpy(), self.npix)
            ss = ss.cpu().numpy()
            for t in range(self.B):
                psnr_.append(p[t])
                ssim_.append(float(ss[t]))
        return psnr_, ssim_


def _log_iterations(denoiser, sched, psnr_all, noise_estimate, logf):
    """Same lines as dvp...online.py:282-304 / :513-535, emitted after the loop (the PSNRs are
    accumulated on the device; reading them per iteration would force a sync per iteration)."""
    for k, nsig in enumerate(sched):
        if (k + 1) % 2 != 0 or k >= len(psnr_all):
            continue
        if not noise_estimate and nsig is not None:
            if nsig < 1:
                msg = '  ADMM-{0} iteration {1: 3d}, sigma {2: 3g}/255, PSNR {3:2.2f} dB.'.format(
                    denoiser.upper(), k + 1, nsig * 255, psnr_all[k])
            else:
                msg = '  ADMM-{0} iteration {1: 3d}, sigma {2: 3g}, PSNR {3:2.2f} dB.'.format(
                    denoiser.upper(), k + 1, nsig, psnr_all[k])
        else:
            msg = '  ADMM-{0} iteration {1: 3d}, PSNR {2:2.2f} dB.'.format(denoiser.upper(), k + 1, psnr_all[k])
        print(msg)
        if logf is not None:
            logf.write(msg + ' \n')


def admm_denoise_bayer_demosaic_pre(y_bayer, Phi_bayer, _lambda=1, gamma=0.01,
                                    denoiser='tv', iter_max=50, noise_estimate=True, sigma=None,
                                    x0_bayer=None,
                                    X_orig=None, model=None, show_iqa=True, demosaic_method='malvar2004', lr_=0.000001,
                                    inital_iter=1, interval_iter=5, logf=None, useGPU=True, device=0, update_=False,
                                    update_per_iter=1, tile=None, return_device=False):
    """Stage 1: ADMM/GAP with the TV prior (warm start).

    y_bayer [H,W], Phi_bayer [H,W,B] float32 numpy.  Returns
    ``(x_bayer_np[H,W,B], psnr_[B], ssim_[B], psnr_all[iters])`` like the reference's
    'tv' branch (:548-549) - the only one ADMM_TV_Warm_Start_save.py reaches - or, for the deep
    branches 'ffdnet_color' / 'fastdvd_color' (:456-500: Malvar demosaic of x - b, plug-in denoiser,
    ONE dual variable), the 6-tuple ``(xbgr3_np, x_bayer_np, psnr_, ssim_, psnr_all, model)`` (:552).
    The reference's 'PPP' branch compares ``denoiser.lower()`` with an upper-case literal (:411) and can
    never be taken.
    ``tile`` (extension, ``parallel.TileContext``, 'tv' only): row-strip tiling of one large frame over the ranks.  Every
    rank passes ITS rows of y / Phi / x0 / X_orig; the TV prior exchanges 8 rows of its input with the neighbouring ranks
    and all-gathers its early-stop energies once per iteration, and the returned arrays are the full frame.
    ``return_device`` (extension, 'tv' only) returns x as a CUDA tensor in the ``x0_bayer`` layout [H,W,B] (tiled: this
    rank's rows) instead of the tuple - a warm start that stage 2 takes without a gather or a host round trip.
    """
    name = denoiser if denoiser == 'tv' else str(denoiser).lower()
    if name in ('ffdnet_color', 'fastdvd_color'):
        if tile is not None or return_device:
            raise NotImplementedError("tiled stage 1 and return_device cover the TV prior; the deep stage-1 branches "
                                      "('%s') run on a whole frame" % name)
        return _stage1_deep(y_bayer, Phi_bayer, _lambda, gamma, name, denoiser, iter_max, noise_estimate, sigma, x0_bayer,
                            X_orig, model, show_iqa, demosaic_method, lr_, inital_iter, interval_iter, logf, update_,
                            update_per_iter)
    if denoiser != 'tv':
        raise ValueError('Unsupported denoiser {}!'.format(denoiser))
    sigma, iter_max = _as_list(sigma, iter_max)
    pb = _Problem(y_bayer, Phi_bayer, x0_bayer, X_orig)
    if tile is not None:
        if pb.H != tile.rows or pb.W != tile.W:
            raise ValueError("tiled mode: pass this rank's rows (%d x %d), got %d x %d" % (tile.rows, tile.W, pb.H, pb.W))
        tile.enable_p2p(pb.B, ops.TV_HALO)                               # the TV halo goes peer to peer over NVLink
        ws = ops.TvStripWorkspace(pb.H, pb.W, pb.B, pb.y.device)
        tv = tile.tv_chambolle
    else:
        ws = ops.TvWorkspace(pb.H, pb.W, pb.B, pb.y.device)
        tv = ops.tv_chambolle
    n_total = int(sum(iter_max))
    want_iqa = bool(show_iqa and X_orig is not None and not return_device)
    sse = torch.zeros(max(n_total, 1), dtype=torch.float64, device=pb.y.device) if want_iqa else None
    b_next = torch.empty_like(pb.b)
    theta, b, x = pb.theta, pb.b, pb.x
    sched = []
    k = 0
    for idx, nsig in enumerate(sigma):
        for _ in range(iter_max[idx]):
            # x = (theta+b) + lambda*At((y - A(theta+b))/(Phi_sum+gamma))            (:389-391) [+ PSNR of x, :507-512]
            ops.project_stage1(theta, b, pb.phi, pb.y, pb.phisum, x, _lambda, gamma,
                               orig=pb.orig if want_iqa else None, sse=sse[k:k + 1] if want_iqa else None)
            # theta = clip(TV(x - b)); b = b - (x - theta)                               (:403-407, :501-503)
            tv(x, b, -1.0, theta, b_next, -1.0, True, ws, weight=0.1, n_iter_max=5)
            b, b_next = b_next, b
            sched.append(nsig)
            k += 1
    if return_device:
        return ops.planar_to_pixlast(x, 1, pb.B).view(pb.H, pb.W, pb.B)
    if tile is not None:                                                # stage 1 returns x, not theta (:538-541)
        return _tiled_outputs(tile, pb, None, x, sse, X_orig, denoiser, sched, noise_estimate, logf, None, None)
    psnr_all = []
    if want_iqa:
        psnr_all = list(iqa.psnr_from_sse(sse.cpu().numpy()[:n_total], pb.npix * pb.B))
        _log_iterations(denoiser, sched, psnr_all, noise_estimate, logf)
    x_bayer_np = pb.to_hwb(x)                                           # stage 1 returns x, not theta (:538-541)
    psnr_, ssim_ = pb.frame_iqa(x, x_bayer_np, X_orig)
    return x_bayer_np, psnr_, ssim_, psnr_all


def _stage1_deep(y_bayer, Phi_bayer, _lambda, gamma, name, denoiser, iter_max, noise_estimate, sigma, x0_bayer, X_orig, model,
                 show_iqa, demosaic_method, lr_, inital_iter, interval_iter, logf, update_, update_per_iter):
    """Deep branches of stage 1 (dvp...online.py:456-503): v = x - b -> Malvar -> denoiser -> theta; b -= x - theta."""
    from . import fastdvdnet_adapter, ffdnet_adapter
    if demosaic_method != 'malvar2004':
        raise ValueError("demosaic_method must be 'malvar2004'")       # anything else leaves x_rgb at zeros in the reference (:451)
    if update_ and name == 'ffdnet_color':
        # the reference passes update_ as ``updata_`` on EVERY iteration here (:467): off the update interval the adapter
        # then returns a (tensor, model) tuple that the sampling below indexes -> TypeError.  Only update_=False runs.
        raise NotImplementedError("stage 1 with ffdnet_color and update_=True fails in the reference itself (dvp...online.py:467); "
                                  "use twoStageAdmm_denoise_bayer for the online-adaptive loop")
    sigma, iter_max = _as_list(sigma, iter_max)
    pb = _Problem(y_bayer, Phi_bayer, x0_bayer, X_orig)
    dev = pb.y.device
    H, W, B = pb.H, pb.W, pb.B
    n_total = int(sum(iter_max))
    want_iqa = bool(show_iqa and X_orig is not None)
    sse = torch.zeros(max(n_total, 1), dtype=torch.float64, device=dev) if want_iqa else None
    theta, b, x = pb.theta, pb.b, pb.x
    x_rgb = torch.empty((B, 3, H, W), dtype=torch.float32, device=dev)
    adapter = ffdnet_adapter if name == 'ffdnet_color' else fastdvdnet_adapter
    sched, k, xhat = [], 0, None
    for idx, nsig in enumerate(sigma):
        for _ in range(iter_max[idx]):
            ops.project_stage1(theta, b, pb.phi, pb.y, pb.phisum, x, _lambda, gamma)             # :389-391
            ops.malvar2004(x, b, -1.0, None, 0.0, x_rgb, None)                                   # x_rgb = Malvar(merge(x - b)) :458-466
            xhat = adapter.denoise_planar(x_rgb, pb, nsig, model, lr_, False, update_per_iter)   # :467-470 / :492
            ops.dual_update_stage1(xhat, x, b, theta, first_iter=(k == 0),
                                   orig=pb.orig if want_iqa else None, sse=sse[k:k + 1] if want_iqa else None)
            sched.append(nsig)
            k += 1
    psnr_all = []
    if want_iqa:
        psnr_all = list(iqa.psnr_from_sse(sse.cpu().numpy()[:n_total], pb.npix * B))
        _log_iterations(denoiser, sched, psnr_all, noise_estimate, logf)
    x_bayer_np = pb.to_hwb(x)                                                                    # stage 1 returns x (:538-541)
    psnr_, ssim_ = pb.frame_iqa(x, x_bayer_np, X_orig)
    xbgr3_np = cuda2np(ops.planar_to_pixlast(xhat, 3, B).view(H, W, 3, B))
    return xbgr3_np, x_bayer_np, psnr_, ssim_, psnr_all, model


class _TileView:
    """What an adapter needs to know about a halo-extended strip: where the own rows sit and how to normalise the loss."""

    def __init__(self, tile, top, ext_rows):
        self.top, self.rows = top, tile.rows
        self.total_pixels, self.H_total = tile.total_pixels, tile.H_total
        self.g0 = tile.r0 - top                      # global row of the first row of the extended strip


def _tiled_demosaic(tile, x, b, inv_rou, w, tau, x_rgb, u, model_demosaic, mosaic):
    """The demosaic step of a row strip (SURVEY 8(e)): DDnet on strips (``DDnetEngine.forward_tiled``: 88 rows of the
    merged mosaic, 40 rows of its temp2 input) or Malvar (2 rows of the merged mosaic), then u = x_rgb - w/tau.  u (own
    rows) is filled in place; returns x_rgb (own rows: ``x_rgb`` itself for Malvar, the engine's buffer for DDnet)."""
    B, rows, W = x.shape
    if model_demosaic is not None:
        from . import ddnet_adapter
        x_rgb = ddnet_adapter._unwrap(model_demosaic).engine().forward_tiled(ops.axpy(x, inv_rou, b, out=mosaic), tile)
    else:
        m_ext, top2 = tile.exchange(ops.axpy(x, inv_rou, b).view(B, 1, rows, W), 2)    # merged mosaic x + b/rho
        rgb_ext = torch.empty((B, 3, m_ext.shape[2], W), dtype=torch.float32, device=x.device)
        ops.malvar2004(m_ext.view(B, m_ext.shape[2], W), None, 0.0, None, 0.0, rgb_ext, None)
        x_rgb.copy_(rgb_ext[:, :, top2:top2 + rows])
    ops.axpy(x_rgb, -float(np.float32(1 / tau)), w, out=u)                              # u = x_rgb - w/tau (:198)
    return x_rgb


def _tiled_denoise(tile, adapter, halo, u, pb, nsig, model, lr_, do_update, update_per_iter, grad_sync):
    """The denoise step of a row strip: `halo` rows of the denoiser input u (own rows), overlap-tile denoising, crop;
    FastDVDnet inference instead exchanges 40 rows per DenBlock.  Returns xhat (own rows)."""
    rows = u.shape[2]
    if adapter.__name__.endswith("fastdvdnet_adapter") and not do_update:
        # inference: one 40-row exchange per DenBlock instead of an 80-row overlap for the whole cascade
        return adapter._unwrap(model).engine().forward_tiled(u, nsig, tile)
    u_ext, top = tile.exchange(u, halo)
    view = _TileView(tile, top, u_ext.shape[2])
    xhat_ext = adapter.denoise_planar(u_ext, pb, nsig, model, lr_, do_update, update_per_iter, grad_sync=grad_sync, tile=view)
    return xhat_ext[:, :, top:top + rows].contiguous()


def _tiled_outputs(tile, pb, xhat, theta, sse, X_orig, denoiser, sched, noise_estimate, logf, model_denoise, model_demosaic):
    """Gather the strips into full-frame results on every rank (``tile.gather_root_only``: on rank 0 only, the others return
    None for the image arrays and an empty SSIM list); PSNR from all-reduced squared errors.  ``theta`` is the Bayer cube
    returned (stage 1 passes x).  Without ``xhat`` (the TV prior) the result is the reference's 4-tuple
    ``(x_bayer_np, psnr_, ssim_, psnr_all)``."""
    B = pb.B
    Ht, W = tile.H_total, tile.W
    psnr_all = []
    if sse is not None:
        tile.all_reduce_sum(sse)
        psnr_all = list(iqa.psnr_from_sse(sse.cpu().numpy()[:len(sched)], Ht * W * B))
        if tile.rank == 0:
            _log_iterations(denoiser, sched, psnr_all, noise_estimate, logf)
    root = bool(tile.gather_root_only)                                      # only rank 0 assembles the frame (others: None)
    timing = os.environ.get("SCI_TILE_TIMING") and tile.rank == 0
    if timing:
        import time
        torch.cuda.synchronize(); t0 = time.time()
    theta_full = tile.gather_rows(theta, root)                              # [B, Ht, W]
    xhat_full = tile.gather_rows(xhat, root) if xhat is not None else None  # [B, 3, Ht, W]
    if timing:
        torch.cuda.synchronize(); t1 = time.time()
    have = theta_full is not None
    x_bayer_np = cuda2np(ops.planar_to_pixlast(theta_full.contiguous(), 1, B).view(Ht, W, B)) if have else None
    xbgr3_np = None
    if have and xhat is not None:
        xbgr3_np = cuda2np(ops.planar_to_pixlast(xhat_full.contiguous(), 3, B).view(Ht, W, 3, B))
    if timing:
        torch.cuda.synchronize(); t2 = time.time()
        print("tiled outputs: gather %.1f ms, remap + device-to-host %.1f ms" % (1e3 * (t1 - t0), 1e3 * (t2 - t1)), file=sys.stderr)
    psnr_, ssim_ = [], []
    if X_orig is not None:
        fsse = torch.zeros(B, dtype=torch.float64, device=theta.device)
        ops.psnr_accum(theta, pb.orig, fsse)
        tile.all_reduce_sum(fsse)
        psnr_ = list(iqa.psnr_from_sse(fsse.cpu().numpy(), Ht * W))
        orig_g = tile.gather_rows(pb.orig, root)
        if orig_g is not None:
            orig_full = cuda2np(ops.planar_to_pixlast(orig_g.contiguous(), 1, B).view(Ht, W, B))
            ssim_ = [iqa.ssim(orig_full[:, :, t], x_bayer_np[:, :, t], data_range=1.) for t in range(B)]
    if xhat is None:
        return x_bayer_np, psnr_, ssim_, psnr_all
    return xbgr3_np, x_bayer_np, psnr_, ssim_, psnr_all, model_denoise, model_demosaic


def twoStageAdmm_denoise_bayer(y_bayer, Phi_bayer, _lambda=1, gamma=0.01,
                               denoiser='tv', iter_max=50, noise_estimate=True, sigma=None,
                               x0_bayer=None,
                               X_orig=None, model_denoise=None, model_demosaic=None, show_iqa=True,
                               demosaic_method='malvar2004', lr_=0.000001,
                               inital_iter=1, interval_iter=5, logf=None, useGPU=True, update_=False, update_per_iter=1,
                               close_form_demosaic=False,
                               large=False, update_times=-1, args=None, grad_sync=None, return_device=False, tile=None):
    """Stage 2: ADMM with a plug-in denoiser ('tv', 'ffdnet_color', 'fastdvd_color') and optional
    online fine-tuning of the denoiser on the measurement-consistency loss.

    Returns the reference's tuples: 'tv' -> ``(x_bayer_np, psnr_, ssim_, psnr_all)`` (:322-323),
    otherwise ``(xbgr3_np[H,W,3,B], x_bayer_np[H,W,B], psnr_, ssim_, psnr_all, model_denoise,
    model_demosaic)`` (:324).  ``grad_sync`` (extension, default None) is a callable applied to the
    flat gradient bucket before each Adam step; the multi-GPU driver passes an NCCL all-reduce.
    ``return_device`` (extension) returns the planar device tensors ``(xhat[B,3,H,W], theta[B,H,W])`` instead of
    numpy arrays (no D2H copy, no host sync) — used by bench.py for the HBM-resident measurement.
    ``tile`` (extension, ``parallel.TileContext``): spatial row-strip tiling of one large frame over the ranks (BASELINE
    config 5).  Every rank passes ITS rows of y / Phi / x0 / X_orig; the mosaic (2 rows for Malvar; for DDnet 88 rows, and
    40 rows of its temp2 input per frame chunk) and the denoiser input (80 rows for FastDVDnet, 28 for FFDNet; 8 rows of the
    TV input and an all-gather of its early-stop energies for 'tv') are halo-exchanged with the neighbouring ranks once per
    iteration, PSNR sums and the fine-tune gradients are all-reduced, and the returned arrays are the full frame (gathered
    on every rank).  The closed-form demosaic is pixel-wise and needs no halo.  DDnet needs strips and a width that are
    multiples of 8, and strips of at least 88 rows over several ranks (ValueError otherwise).

    Reproducibility: the fine-tune's backward reductions (weight gradients, bias / BatchNorm column sums) run in a fixed
    order, so the same inputs, the same numpy / torch seeds (``utilspy.worker_init_fn``), the same GPU model and the same
    world size and transport give bit-identical reconstructions (``xbgr3``, ``x_bayer`` / ``theta``) and bit-identical fine-tuned weights.  Not covered: NCCL's
    all-reduce in ``grad_sync`` (its algorithm choice; gloo is deterministic), DDnet's self-supervised update (never
    run by the solvers), and the printed fp64 diagnostics (PSNR, SSIM, losses), which may vary at ~1e-16 relative.
    """
    name = denoiser if denoiser == 'tv' else str(denoiser).lower()
    if name not in ('tv', 'ffdnet_color', 'fastdvd_color'):
        raise ValueError('Unsupported denoiser {}!'.format(denoiser))
    sigma, iter_max = _as_list(sigma, iter_max)
    if tile is not None and name != 'tv' and model_demosaic is not None:
        from .engine import DDnetEngine
        DDnetEngine.check_tile(tile)                                   # strips DDnet cannot run on: refused before GPU work
    pb = _Problem(y_bayer, Phi_bayer, x0_bayer, X_orig)
    dev = pb.y.device
    H, W, B = pb.H, pb.W, pb.B
    if tile is not None:
        if H != tile.rows or W != tile.W:
            raise ValueError("tiled mode: pass this rank's rows (%d x %d), got %d x %d" % (tile.rows, tile.W, H, W))
        if name == 'tv':
            tile.enable_p2p(B, ops.TV_HALO)                                # 8 rows of the TV input, peer to peer
        else:
            if grad_sync is None:
                grad_sync = tile.all_reduce_sum      # loss is normalised by the whole frame -> gradients ADD over strips
            exchanges = [(3 * B, 28 if name == 'ffdnet_color' else 80)]    # (planes, rows) of the largest exchanges
            if model_demosaic is not None:
                bc = DDnetEngine.tiled_chunk_frames(B, tile)
                exchanges += [(B, DDnetEngine.STAGE_A_HALO), (2 * bc * 32, DDnetEngine.STAGE_B_HALO)]
            tile.enable_p2p(*max(exchanges, key=lambda e: e[0] * e[1]))   # boundary rows go peer to peer over NVLink
    alpha = 0.01 if name == 'tv' else 1                                  # :101-104
    rou = 0.55 if name == 'fastdvd_color' else 1                         # :106-109
    tau = 100                                                            # :110
    if close_form_demosaic:                                              # :112-118
        tau, rou = 10, 0.55
    inv_rou = float(np.float32(1 / rou))
    n_total = int(sum(iter_max))
    want_iqa = bool(show_iqa and X_orig is not None)
    sse = torch.zeros(max(n_total, 1), dtype=torch.float64, device=dev) if want_iqa else None
    theta, b, x = pb.theta, pb.b, pb.x
    xhat = None
    if name == 'tv':
        ws = ops.TvWorkspace(H, W, B, dev) if tile is None else ops.TvStripWorkspace(H, W, B, dev)
        tv = ops.tv_chambolle if tile is None else tile.tv_chambolle
        b_next = torch.empty_like(b)
    else:
        from . import ddnet_adapter, fastdvdnet_adapter, ffdnet_adapter
        mosaic = torch.empty_like(x) if model_demosaic is not None else None
        w = torch.zeros((B, 3, H, W), dtype=torch.float32, device=dev)
        x_rgb = torch.empty_like(w)
        u = torch.empty_like(w)
        if demosaic_method != 'malvar2004':
            # In the reference every other value silently leaves x_rgb at zeros (``.lower`` is compared
            # unbound, :187,:233 — SURVEY App. D.2); that degenerate loop is refused rather than reproduced.
            raise ValueError("demosaic_method must be 'malvar2004'")
    sched = []
    k = 0
    update_i = 0
    if name == 'fastdvd_color' and update_:
        # The FastDVDnet fine-tune perturbs its input with HOST numpy-RNG noise (utils_image.py:183-192); a helper
        # thread keeps those draws ahead of the GPU with exact global-RNG semantics (fastdvdnet_adapter.NoiseStream).
        # (tiled mode: every rank draws the noise of the WHOLE frame and cuts its rows out, so that is the shape to run ahead with)
        fastdvdnet_adapter.noise_stream.prefetch((B, 3, tile.H_total if tile is not None else H, W))
    for idx, nsig in enumerate(sigma):
        for _ in range(iter_max[idx]):
            # p = theta - b/rho ; x = p + Phi*((y - A p)/(alpha*rho + Phi_sum))                     (:128-140)
            ops.project_stage2(theta, b, pb.phi, pb.y, pb.phisum, x, alpha, rou)
            if name == 'tv':
                # theta = clip(TV(x + b/rho)); b = b + (x - theta)                                   (:153-160, :265-267)
                tv(x, b, inv_rou, theta, b_next, 1.0, True, ws, weight=0.1, n_iter_max=5)
                b, b_next = b_next, b
                if want_iqa:
                    ops.psnr_accum(theta.view(1, -1), pb.orig.view(1, -1), sse[k:k + 1])
            else:
                # x_rgb = Malvar(merge(x + b/rho)) for all frames ; u = x_rgb - w/tau                 (:169-198)
                do_update = bool(update_ and k > inital_iter and k % interval_iter == 0)
                if name == 'fastdvd_color':
                    do_update = do_update and (update_i < update_times or update_times < 0)   # :247
                    update_i += int(do_update)
                adapter = ffdnet_adapter if name == 'ffdnet_color' else fastdvdnet_adapter
                if close_form_demosaic and k > 0:
                    # x_rgb = (rho*x3 + b3 + tau*xhat + w) / (rho*mask + tau) [clip for FFDNet] ; u = x_rgb - w/tau   (:175-182)
                    # (pixel-wise: on a strip its own rows, the Bayer phase kept by rows % 4 == 0)
                    ops.closed_form_demosaic(x, b, xhat, w, rou, tau, name == 'ffdnet_color', x_rgb, u)
                elif tile is not None:
                    x_rgb = _tiled_demosaic(tile, x, b, inv_rou, w, tau, x_rgb, u, model_demosaic, mosaic)
                elif model_demosaic is not None:
                    # deep demosaicking: x_rgb = DDnet(merge(x + b/rho)) ; u = x_rgb - w/tau          (:192-198, :241-246)
                    x_rgb = ddnet_adapter.demosaic_planar(ops.axpy(x, inv_rou, b, out=mosaic), model_demosaic)
                    ops.axpy(x_rgb, -float(np.float32(1 / tau)), w, out=u)
                else:
                    ops.malvar2004(x, b, inv_rou, w, 1 / tau, x_rgb, u)
                if tile is None:
                    xhat = adapter.denoise_planar(u, pb, nsig, model_denoise, lr_, do_update, update_per_iter,
                                                  grad_sync=grad_sync)
                else:
                    xhat = _tiled_denoise(tile, adapter, 28 if name == 'ffdnet_color' else 80, u, pb, nsig, model_denoise,
                                          lr_, do_update, update_per_iter, grad_sync)
                # theta = clip(RGGB samples of xhat) ; b += x - theta ; w += x_rgb - xhat [+ PSNR]    (:206-209, :265-280)
                ops.dual_update_rgb(xhat, x_rgb, w, x, b, theta, first_iter=(k == 0),
                                    orig=pb.orig if want_iqa else None, sse=sse[k:k + 1] if want_iqa else None)
            sched.append(nsig)
            k += 1
    if return_device:
        return xhat, theta
    if tile is not None:
        return _tiled_outputs(tile, pb, xhat, theta, sse if want_iqa else None, X_orig, denoiser, sched, noise_estimate,
                              logf, model_denoise, model_demosaic)
    psnr_all = []
    if want_iqa:
        psnr_all = list(iqa.psnr_from_sse(sse.cpu().numpy()[:n_total], pb.npix * B))
        _log_iterations(denoiser, sched, psnr_all, noise_estimate, logf)
    elif X_orig is None and logf is not None:
        for kk, nsig in enumerate(sched):                                                        # :307-309
            if (kk + 2) % 2 == 0 and nsig is not None:
                logf.write('  ADMM-{0} iteration {1: 3d}, sigma {2: 3g}/255 \n'.format(denoiser.upper(), kk + 2, nsig * 255))
    x_bayer_np = pb.to_hwb(theta)                                        # stage 2 returns theta (:312-315)
    psnr_, ssim_ = pb.frame_iqa(theta, x_bayer_np, X_orig)
    if name == 'tv':
        return x_bayer_np, psnr_, ssim_, psnr_all
    xbgr3_np = cuda2np(ops.planar_to_pixlast(xhat, 3, B).view(H, W, 3, B))
    return xbgr3_np, x_bayer_np, psnr_, ssim_, psnr_all, model_denoise, model_demosaic


def twoStageAdmm_denoise_gray(y, Phi, denoiser='ffdnet_gray', iter_max=50, sigma=None, x0=None, X_orig=None,
                              model_denoise=None, show_iqa=True, lr_=0.000001, inital_iter=1, interval_iter=5, logf=None,
                              update_=False, update_per_iter=1, noise_estimate=False, grad_sync=None, update_times=-1):
    """Two-stage ADMM with an online-adapted deep denoiser on a GRAYSCALE cube: 'ffdnet_gray' (BASELINE config 2) or
    'fastdvd_gray' (the grayscale video SCI case of adaptive PnP with FastDVDnet, ``fastdvdnet_models.FastDVDnet`` with
    ``num_color_channels=1``).

    The reference has no function for either (``twoStageAdmm_denoise_bayer`` only knows 'tv', 'ffdnet_color' and
    'fastdvd_color', dvp...online.py:147,164,214,262; the gray network is only constructed by the script's ``else``
    branch, two_stage_ADMM_Online_FFD_Warm.py:37-40).  Following SURVEY §8(c) this is the SAME loop with the Bayer split /
    demosaic replaced by the identity and every constant the colour branch uses for the same denoiser: tau = 100, k = 0
    aliasing included, alpha = 1 and rho = 1 for 'ffdnet_gray', rho = 0.55 for 'fastdvd_gray' (dvp:101-109), whose
    fine-tune is ``fastdvdnet_denoiser_full_tensor_v2`` with one plane (noise (B,1,H,W) from the global numpy RNG, loss
    MSE(sum_t xhat_t Phi_t, y)) and is limited by ``update_times`` (dvp:247; 'ffdnet_gray' ignores it).  Parity is checked
    against the derived oracles (``oracle.admm.twoStageAdmm_denoise_gray`` for 'ffdnet_gray',
    ``oracle.gray_fastdvd.twoStageAdmm_denoise_gray`` for 'fastdvd_gray') and reported as "parity vs derived oracle".
    'fastdvd_gray' needs H and W multiples of 4 (ValueError before any GPU work).

    Reproducibility: the fine-tune's backward reductions (weight gradients, bias / BatchNorm column sums) run in a fixed
    order, so the same inputs, the same numpy / torch seeds (``utilspy.worker_init_fn``), the same GPU model and the same
    world size and transport give bit-identical reconstructions (``xhat``, ``theta``) and bit-identical fine-tuned weights.  Not covered: NCCL's
    all-reduce in ``grad_sync`` (its algorithm choice; gloo is deterministic), DDnet's self-supervised update (never
    run by the solvers), and the printed fp64 diagnostics (PSNR, SSIM, losses), which may vary at ~1e-16 relative.

    y [H,W], Phi [H,W,B], x0 [H,W,B] (warm start) -> (xhat_np[H,W,B], theta_np[H,W,B], psnr_, ssim_, psnr_all, model)."""
    name = str(denoiser).lower()
    if name not in ('ffdnet_gray', 'fastdvd_gray'):
        raise ValueError('Unsupported denoiser {}!'.format(denoiser))
    if name == 'fastdvd_gray' and (y.shape[0] % 4 or y.shape[1] % 4):
        raise ValueError("'fastdvd_gray' needs H and W multiples of 4 (the native FastDVDnet engine), got %d x %d"
                         % (y.shape[0], y.shape[1]))
    from . import fastdvdnet_adapter, ffdnet_adapter
    adapter = ffdnet_adapter if name == 'ffdnet_gray' else fastdvdnet_adapter
    sigma, iter_max = _as_list(sigma, iter_max)
    pb = _Problem(y, Phi, x0, X_orig)
    dev = pb.y.device
    H, W, B = pb.H, pb.W, pb.B
    rou = 0.55 if name == 'fastdvd_gray' else 1                                       # dvp:106-109
    inv_rou = float(np.float32(1 / rou))
    tau = 100
    n_total = int(sum(iter_max))
    want_iqa = bool(show_iqa and X_orig is not None)
    sse = torch.zeros(max(n_total, 1), dtype=torch.float64, device=dev) if want_iqa else None
    theta, b, x = pb.theta, pb.b, pb.x
    w = torch.zeros((B, 1, H, W), dtype=torch.float32, device=dev)
    x_pre = torch.empty((B, H, W), dtype=torch.float32, device=dev)
    u = torch.empty((B, 1, H, W), dtype=torch.float32, device=dev)
    if name == 'fastdvd_gray' and update_:
        fastdvdnet_adapter.noise_stream.prefetch((B, 1, H, W))                        # see twoStageAdmm_denoise_bayer
    sched, k, xhat, update_i = [], 0, None, 0
    for idx, nsig in enumerate(sigma):
        for _ in range(iter_max[idx]):
            ops.project_stage2(theta, b, pb.phi, pb.y, pb.phisum, x, 1, rou)              # alpha = 1
            ops.axpy(x, inv_rou, b, out=x_pre)                                            # x + b/rho
            ops.axpy(x_pre.view(B, 1, H, W), -float(np.float32(1 / tau)), w, out=u)       # - w/tau
            do_update = bool(update_ and k > inital_iter and k % interval_iter == 0)
            if name == 'fastdvd_gray':
                do_update = do_update and (update_i < update_times or update_times < 0)   # dvp:247
                update_i += int(do_update)
            xhat = adapter.denoise_planar(u, pb, nsig, model_denoise, lr_, do_update, update_per_iter, grad_sync=grad_sync)
            _lib_call("sci_dual_update_gray", xhat, x_pre, w, x, b, theta, k == 0, pb.orig if want_iqa else None,
                      sse[k:k + 1] if want_iqa else None)
            sched.append(nsig)
            k += 1
    psnr_all = []
    if want_iqa:
        psnr_all = list(iqa.psnr_from_sse(sse.cpu().numpy()[:n_total], pb.npix * B))
        _log_iterations(denoiser, sched, psnr_all, noise_estimate, logf)
    theta_np = pb.to_hwb(theta)
    psnr_, ssim_ = pb.frame_iqa(theta, theta_np, X_orig)
    xhat_np = pb.to_hwb(xhat.view(B, H, W))
    return xhat_np, theta_np, psnr_, ssim_, psnr_all, model_denoise


def _lib_call(name, xhat, x_pre, w, x, b, theta, first, orig, sse):
    from ._lib import call, ptr, stream
    call(name, ptr(xhat), ptr(x_pre), ptr(w), ptr(x), ptr(b), ptr(theta), int(bool(first)), theta.numel(), ptr(orig), ptr(sse),
         stream())
