"""Oracle: grayscale two-stage ADMM with online FastDVDnet (the product's ``twoStageAdmm_denoise_gray(denoiser='fastdvd_gray')``).

Test infrastructure.  DERIVED restatements — the reference has no grayscale FastDVDnet loop (``twoStageAdmm_denoise_bayer``
knows 'tv', 'ffdnet_color' and 'fastdvd_color' only, dvp...online.py:147,164,214,262), and the reference's gray branch of
``fastdvdnet_denoiser_full_tensor_v2`` is not restated here.  The rule is that of BASELINE config 2 (SURVEY §8(c),
``admm.twoStageAdmm_denoise_gray``): the colour loop with the Bayer split and demosaic replaced by the identity, every
constant the one the colour branch uses for the same denoiser.  Parity against these is "parity vs derived oracle".
"""
import numpy as np
import torch
import torch.nn as nn

from .adapters import NUM_IN_FR_EXT, fastdvdnet_seqdenoise
from .admm import _final_iqa, _listify
from .iqa import compare_psnr
from .sci_ops import A_


def fastdvdnet_gray_denoise_full_tensor(x, y, Phi, sigma, model, lr_=1e-6, updata_=False, update_per_iter=1, losses=None):
    """``adapters.fastdvdnet_denoiser_full_tensor_v2`` (test_fastdvdnet.py:325-500) with one plane and the Bayer sampling
    removed: x [H,W,B] gray cube, y [H,W], Phi [H,W,B], ``model`` the single-channel FastDVDnet (``networks.FastDVDnet(5, 1)``,
    optionally wrapped).  With ``updata_``: training input x + float32(float64(x) + N(0,(5/255)^2)), the noise drawn ONCE per
    call from the global numpy RNG with shape (B,1,H,W); BatchNorm frozen (eval) but its affine parameters trained; a fresh
    Adam per (lr, n_iter) pair; loss MSE(sum_t xhat_t * Phi_t, y) over H*W; the final denoise of the CLEAN input ->
    ``(outv[H,W,B], model)``.  Without: ``outv[H,W,B]``."""
    noisestd = torch.FloatTensor([sigma])
    v = x.permute(2, 0, 1).unsqueeze(1)                                  # [B,1,H,W]
    net = model.module if hasattr(model, "module") else model
    if updata_:
        n_update_iter, lr_all = ([update_per_iter], [lr_]) if isinstance(update_per_iter, int) else (update_per_iter, lr_)
        mse = nn.MSELoss()
        noise = np.random.normal(0, 5 / 255, tuple(v.shape))
        v_plus = v + torch.from_numpy(v.detach().numpy() + noise).float()
        model.train()
        for m in net.modules():
            if isinstance(m, nn.BatchNorm2d):
                m.eval()
        for lr_i, nit in zip(lr_all, n_update_iter):
            opt = torch.optim.Adam(filter(lambda p: p.requires_grad, model.parameters()), lr=lr_i)
            for _ in range(nit):
                N, C, H, W = v.shape
                noise_map = noisestd.expand((1, 1, H, W))
                frames = []
                for f in range(N):
                    idx = (torch.arange(f, f + NUM_IN_FR_EXT) - 2) % N
                    frames.append(model(v_plus[idx].reshape((1, -1, H, W)), noise_map)[0, 0])
                outv = torch.stack(frames, 2)                              # [H,W,B]
                loss = mse(torch.sum(outv * Phi, dim=2), y)
                opt.zero_grad()
                loss.backward()
                opt.step()
                if losses is not None:
                    losses.append(float(loss.detach()))
        with torch.no_grad():
            outv = fastdvdnet_seqdenoise(v, noisestd, NUM_IN_FR_EXT, model)[:, 0].permute(1, 2, 0)
            if losses is not None:
                losses.append(float(mse(torch.sum(outv * Phi, dim=2), y)))
        return outv, model
    model.eval()
    with torch.no_grad():
        return fastdvdnet_seqdenoise(v, noisestd, NUM_IN_FR_EXT, model)[:, 0].permute(1, 2, 0)


def twoStageAdmm_denoise_gray(y, Phi, denoiser='fastdvd_gray', iter_max=50, sigma=None, x0=None, X_orig=None,
                              model_denoise=None, show_iqa=True, lr_=1e-6, inital_iter=1, interval_iter=5, update_=False,
                              update_per_iter=1, update_times=-1, trace=None):
    """The gray loop of ``admm.twoStageAdmm_denoise_gray`` with online FastDVDnet-gray and the constants of the colour
    FastDVDnet branch (dvp:101-110): alpha = 1, rho = 0.55, tau = 100,
        p = theta - b/rho ; x = p + Phi*((y - A p)/(alpha*rho + Phi_sum))
        x_pre = x + b/rho ; xhat = FastDVDnet_gray(x_pre - w/tau) [online fine-tune] ; theta = clip(xhat)
        b += x - theta ; w += x_pre - xhat
    including the k = 0 aliasing of xall/theta_all; the update trigger is
    ``update_ and k > inital_iter and k % interval_iter == 0 and (update_i < update_times or update_times < 0)`` (:200, :247).
    Returns (xhat_np[H,W,B], theta_np[H,W,B], psnr_, ssim_, psnr_all, model)."""
    if str(denoiser).lower() != 'fastdvd_gray':
        raise ValueError('Unsupported denoiser {}!'.format(denoiser))
    y = torch.from_numpy(np.ascontiguousarray(y))
    Phi = torch.from_numpy(np.ascontiguousarray(Phi))
    sigma, iter_max = _listify(sigma, iter_max)
    Phi_sum = torch.sum(Phi, dim=2)
    Phi_sum[Phi_sum == 0] = 1
    x0all = (y.unsqueeze(2) * Phi) if x0 is None else x0.clone()
    xall = x0all
    theta = x0all
    ball = torch.zeros_like(x0all)
    w = torch.zeros_like(x0all)
    alpha, rou, tau = 1, 0.55, 100
    psnr_all, k, update_i = [], 0, 0
    xhat = None
    for idx, nsig in enumerate(sigma):
        for it in range(iter_max[idx]):
            p = theta - (1 / rou) * ball
            t = (y - A_(p, Phi)) / (alpha * rou + Phi_sum)
            xall[...] = p + Phi * t.unsqueeze(2)                       # in place: aliases theta at k = 0
            x_pre = xall + (1 / rou) * ball
            x_w = x_pre - (1 / tau) * w
            do_update = update_ and k > inital_iter and k % interval_iter == 0
            losses = None if trace is None else trace.setdefault('losses', [])
            if do_update and (update_i < update_times or update_times < 0):
                xhat, model_denoise = fastdvdnet_gray_denoise_full_tensor(x_w, y, Phi, nsig, model_denoise, lr_, True,
                                                                          update_per_iter, losses=losses)
                update_i += 1
            else:
                xhat = fastdvdnet_gray_denoise_full_tensor(x_w, y, Phi, nsig, model_denoise, lr_)
            theta[...] = xhat                                          # writes into xall too while they alias (k = 0)
            theta = torch.clip(theta, 0, 1)
            ball = ball + (xall - theta)
            w = w + (x_pre - xhat)
            if show_iqa and X_orig is not None:
                psnr_all.append(compare_psnr(X_orig, theta.numpy(), data_range=1.))
            k += 1
    theta_np = theta.numpy()
    psnr_, ssim_ = _final_iqa(X_orig, theta_np, Phi.shape[2])
    return xhat.detach().numpy(), theta_np, psnr_, ssim_, psnr_all, model_denoise
