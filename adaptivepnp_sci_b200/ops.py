"""Thin tensor-level wrappers over the C ABI (planar device layouts).

Every function launches hand-written sm_100a kernels on the current CUDA stream
through ``_lib``; nothing here computes with PyTorch ops.  Layouts: Bayer-domain
cubes ``[B,H,W]``, RGB cubes ``[B,3,H,W]``, planes ``[H,W]`` (see
``include/sci_b200.h``).
"""
import ctypes

import torch

from . import _lib
from ._lib import call, ptr, require_cuda_f32, stream


def pixlast_to_planar(t_in, C, B):
    """[P..., C, B] (reference pixel-last) -> [B, C, P...] planar.  Bit-exact remap."""
    require_cuda_f32(t_in)
    P = t_in.numel() // (C * B)
    out = torch.empty((B, C, P), dtype=torch.float32, device=t_in.device)
    call("sci_pixlast_to_planar", ptr(t_in), ptr(out), P, C, B, stream())
    return out


def planar_to_pixlast(t_in, C, B):
    """[B, C, P] planar -> [P, C, B] pixel-last.  Bit-exact remap."""
    require_cuda_f32(t_in)
    P = t_in.numel() // (C * B)
    out = torch.empty((P, C, B), dtype=torch.float32, device=t_in.device)
    call("sci_planar_to_pixlast", ptr(t_in), ptr(out), P, C, B, stream())
    return out


def bayer_split_init(y, phi_hwb, x0_hwb=None):
    """K0.  y [H,W], phi_hwb [H,W,B], optional warm start x0_hwb [H,W,B] ->
    (phi [B,H,W], phisum [H,W], theta0 [B,H,W])."""
    require_cuda_f32(y, phi_hwb, x0_hwb)
    H, W, B = phi_hwb.shape
    dev = y.device
    phi = torch.empty((B, H, W), dtype=torch.float32, device=dev)
    phisum = torch.empty((H, W), dtype=torch.float32, device=dev)
    theta0 = torch.empty((B, H, W), dtype=torch.float32, device=dev)
    call("sci_bayer_split_init", ptr(y), ptr(phi_hwb), ptr(x0_hwb), ptr(phi), ptr(phisum), ptr(theta0), H, W, B, stream())
    return phi, phisum, theta0


def project_stage1(theta, b, phi, y, phisum, x_out, lambda_, gamma, orig=None, sse=None):
    require_cuda_f32(theta, b, phi, y, phisum, x_out, orig)
    B = phi.shape[0]
    npix = y.numel()
    call("sci_project_stage1", ptr(theta), ptr(b), ptr(phi), ptr(y), ptr(phisum), ptr(x_out), npix, B,
         float(lambda_), float(gamma), ptr(orig), ptr(sse), stream())
    return x_out


def project_stage2(theta, b, phi, y, phisum, x_out, alpha, rho):
    require_cuda_f32(theta, b, phi, y, phisum, x_out)
    B = phi.shape[0]
    npix = y.numel()
    call("sci_project_stage2", ptr(theta), ptr(b), ptr(phi), ptr(y), ptr(phisum), ptr(x_out), npix, B,
         float(alpha), float(rho), stream())
    return x_out


class TvWorkspace:
    """Scratch for sci_tv_chambolle2d (per-block energy partials + stop indices)."""

    def __init__(self, H, W, B, device):
        self.nbytes = int(_lib.lib.sci_tv_workspace_bytes(H, W, B))
        self.buf = torch.empty(self.nbytes, dtype=torch.uint8, device=device)
        self.shape = (H, W, B)


def tv_chambolle(x, b, c_b, theta_out, b_out, s_b, clip, ws, weight=0.1, eps=2.0e-4, n_iter_max=5, nstop_out=None):
    """K4 fused:  theta = [clip] TV(x + c_b*b);  b_out = b + s_b*(x - theta).  b/b_out may be None."""
    require_cuda_f32(x, b, theta_out, b_out)
    B, H, W = x.shape
    assert ws.shape == (H, W, B)
    call("sci_tv_chambolle2d", ptr(x), ptr(b), float(c_b), ptr(theta_out), ptr(b_out), float(s_b), int(bool(clip)),
         H, W, B, float(weight), float(eps), int(n_iter_max), ptr(ws.buf), ctypes.c_size_t(ws.nbytes),
         ptr(nstop_out), stream())
    return theta_out


TV_HALO = 8          # rows of f = x + c_b*b a TV row strip needs from each neighbour


class TvStripWorkspace:
    """Scratch for sci_tv_strip_main / _finish (per-block energy partials + stop indices) and this strip's energy sums
    ``esum`` [4B, 8] float64, the tensor the ranks gather between the two halves."""

    def __init__(self, rows, W, B, device):
        self.nbytes = int(_lib.lib.sci_tv_strip_workspace_bytes(rows, W, B))
        self.buf = torch.empty(self.nbytes, dtype=torch.uint8, device=device)
        self.esum = torch.empty((4 * B, 8), dtype=torch.float64, device=device)
        self.shape = (rows, W, B)


def _vp(p):
    """Raw device address (int) or None -> ctypes pointer."""
    return ctypes.c_void_p(p) if p else None


def tv_strip_main(x, b, c_b, theta_out, b_out, s_b, clip, ws, row0, H_total, halo_top=None, halo_bot=None, weight=0.1,
                  eps=2.0e-4, n_iter_max=5, flag_top=None, flag_bot=None, seq=0, err=None):
    """Main pass of the TV prior on the row strip x [B, rows, W] (global rows row0 ..) + its energy sums (-> ``ws.esum``).
    halo_top / halo_bot: [B, 8, W] tensors of f, or raw device addresses (peer-to-peer slots, with their flag words)."""
    require_cuda_f32(x, b, theta_out, b_out)
    B, rows, W = x.shape
    assert ws.shape == (rows, W, B)
    ht = ptr(halo_top) if torch.is_tensor(halo_top) else _vp(halo_top)
    hb = ptr(halo_bot) if torch.is_tensor(halo_bot) else _vp(halo_bot)
    call("sci_tv_strip_main", ptr(x), ptr(b), float(c_b), ptr(theta_out), ptr(b_out), float(s_b), int(bool(clip)),
         rows, W, B, int(row0), int(H_total), ht, hb, _vp(flag_top), _vp(flag_bot), int(seq), _vp(err), float(weight),
         float(eps), int(n_iter_max), ptr(ws.buf), ctypes.c_size_t(ws.nbytes), ptr(ws.esum), stream())
    return ws.esum


def tv_strip_finish(x, b, c_b, theta_out, b_out, s_b, clip, ws, row0, H_total, esum_all, halo_top=None, halo_bot=None,
                    weight=0.1, eps=2.0e-4, n_iter_max=5, nstop_out=None):
    """Stop decision from esum_all [world, 4B, 8] (summed in strip order) + the fix-up pass of the channels that stop early."""
    require_cuda_f32(x, b, theta_out, b_out)
    B, rows, W = x.shape
    assert ws.shape == (rows, W, B)
    assert esum_all.is_cuda and esum_all.dtype == torch.float64 and esum_all.is_contiguous() and esum_all.shape[-2:] == (4 * B, 8)
    ht = ptr(halo_top) if torch.is_tensor(halo_top) else _vp(halo_top)
    hb = ptr(halo_bot) if torch.is_tensor(halo_bot) else _vp(halo_bot)
    world = esum_all.numel() // (4 * B * 8)
    call("sci_tv_strip_finish", ptr(x), ptr(b), float(c_b), ptr(theta_out), ptr(b_out), float(s_b), int(bool(clip)),
         rows, W, B, int(row0), int(H_total), ht, hb, float(weight), float(eps), int(n_iter_max), ptr(ws.buf),
         ctypes.c_size_t(ws.nbytes), ptr(esum_all), world, ptr(nstop_out), stream())
    return theta_out


def halo_send_tv(x, b, c_b, up_dst, down_dst, up_flag, down_flag, seq, done, halo=TV_HALO):
    """f = x + c_b*b of the first / last ``halo`` rows of x [B, rows, W] -> the neighbours' slots (raw peer addresses or
    None), then release ``seq`` into their flag words (``done``: the kernel's completion counter, raw address)."""
    require_cuda_f32(x, b)
    B, rows, W = x.shape
    call("sci_halo_send_tv", ptr(x), ptr(b), float(c_b), B, rows, W, int(halo), _vp(up_dst), _vp(down_dst), _vp(up_flag),
         _vp(down_flag), int(seq), _vp(done), stream())


def malvar2004(x, b, c_b, w, inv_tau, x_rgb_out, u_out):
    """K6.  mosaic = x + c_b*b (b may be None) -> x_rgb [B,3,H,W]; u = x_rgb - inv_tau*w (if w given)."""
    require_cuda_f32(x, b, w, x_rgb_out, u_out)
    B, H, W = x.shape
    call("sci_malvar2004", ptr(x), ptr(b), float(c_b), ptr(w), float(inv_tau), ptr(x_rgb_out), ptr(u_out), H, W, B,
         stream())
    return x_rgb_out, u_out


def dual_update_rgb(xhat, x_rgb, w, x, b, theta, first_iter, orig=None, sse=None):
    """K3/K5 fused, in place on (w, b, theta)."""
    require_cuda_f32(xhat, x_rgb, w, x, b, theta, orig)
    B, H, W = x.shape
    call("sci_dual_update_rgb", ptr(xhat), ptr(x_rgb), ptr(w), ptr(x), ptr(b), ptr(theta), int(bool(first_iter)),
         H, W, B, ptr(orig), ptr(sse), stream())


def dual_update_stage1(xhat, x, b, theta, first_iter, orig=None, sse=None):
    """Stage-1 deep branches: theta = clip(samples(xhat)), b -= x - theta, PSNR of x (dvp:439-512); in place."""
    require_cuda_f32(xhat, x, b, theta, orig)
    B, H, W = x.shape
    call("sci_dual_update_stage1", ptr(xhat), ptr(x), ptr(b), ptr(theta), int(bool(first_iter)), H, W, B, ptr(orig), ptr(sse),
         stream())


def closed_form_demosaic(x, b, xhat, w, rho, tau, clip, x_rgb_out, u_out):
    """x_rgb = (rho*x3 + b3 + tau*xhat + w) / (rho*mask + tau) [clip]; u = x_rgb - w/tau  (dvp:175-182, 198)."""
    require_cuda_f32(x, b, xhat, w, x_rgb_out, u_out)
    B, H, W = x.shape
    import numpy as np
    call("sci_closed_form_demosaic", ptr(x), ptr(b), ptr(xhat), ptr(w), float(rho), float(tau), float(np.float32(1 / tau)),
         int(bool(clip)), ptr(x_rgb_out), ptr(u_out), H, W, B, stream())
    return x_rgb_out, u_out


def rgb_to_bayer(rgb):
    require_cuda_f32(rgb)
    B, _, H, W = rgb.shape
    out = torch.empty((B, H, W), dtype=torch.float32, device=rgb.device)
    call("sci_rgb_to_bayer", ptr(rgb), ptr(out), H, W, B, stream())
    return out


def bayer_to_rgb_sparse(mosaic):
    require_cuda_f32(mosaic)
    B, H, W = mosaic.shape
    out = torch.empty((B, 3, H, W), dtype=torch.float32, device=mosaic.device)
    call("sci_bayer_to_rgb_sparse", ptr(mosaic), ptr(out), H, W, B, stream())
    return out


def psnr_accum(a, orig, sse_per_frame):
    """sse_per_frame[t] += sum (a[t]-orig[t])^2  (float64 [B] device tensor)."""
    require_cuda_f32(a, orig)
    B = a.shape[0]
    npix = a.numel() // B
    call("sci_psnr_accum", ptr(a), ptr(orig), npix, B, ptr(sse_per_frame), stream())


def ssim_frames(a, orig):
    """Per-frame SSIM (skimage defaults, float64) of a [B,H,W] against orig [B,H,W], computed on the device -> [B] float64."""
    require_cuda_f32(a, orig)
    B, H, W = a.shape
    acc = torch.zeros(B, dtype=torch.float64, device=a.device)
    call("sci_ssim_accum", ptr(a), ptr(orig), H, W, B, 1.0, ptr(acc), stream())
    return acc / float((H - 6) * (W - 6))


def pad_to_multiple(t, m):
    """[..., H, W] -> reflect-padded (right / bottom, like F.pad(mode='reflect')) to multiples of m; returns (padded, H, W)."""
    require_cuda_f32(t)
    H, W = t.shape[-2:]
    Ho, Wo = (H + m - 1) // m * m, (W + m - 1) // m * m
    if (Ho, Wo) == (H, W):
        return t, H, W
    out = torch.empty(t.shape[:-2] + (Ho, Wo), dtype=torch.float32, device=t.device)
    call("sci_reflect_pad2d", ptr(t.contiguous()), ptr(out), t.numel() // (H * W), H, W, Ho, Wo, stream())
    return out, H, W


def replicate_pad_to_even(t):
    """[..., H, W] -> replication-padded (right / bottom) to even H, W (network_ffdnet.py:56-59); returns (padded, H, W)."""
    require_cuda_f32(t)
    H, W = t.shape[-2:]
    Ho, Wo = H + (H & 1), W + (W & 1)
    if (Ho, Wo) == (H, W):
        return t, H, W
    out = torch.empty(t.shape[:-2] + (Ho, Wo), dtype=torch.float32, device=t.device)
    call("sci_replicate_pad2d", ptr(t.contiguous()), ptr(out), t.numel() // (H * W), H, W, Ho, Wo, stream())
    return out, H, W


def crop_to(t, Hc, Wc):
    """[..., H, W] -> contiguous [..., Hc, Wc] (top-left crop)."""
    require_cuda_f32(t)
    H, W = t.shape[-2:]
    if (Hc, Wc) == (H, W):
        return t
    out = torch.empty(t.shape[:-2] + (Hc, Wc), dtype=torch.float32, device=t.device)
    call("sci_crop2d", ptr(t.contiguous()), ptr(out), t.numel() // (H * W), H, W, Hc, Wc, stream())
    return out


def axpy(x, a, y, out=None):
    """out = x + a*y (elementwise, fp32)."""
    require_cuda_f32(x, y, out)
    if out is None:
        out = torch.empty_like(x)
    call("sci_axpy", ptr(x), float(a), ptr(y), ptr(out), x.numel(), stream())
    return out
