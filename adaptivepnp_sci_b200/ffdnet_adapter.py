"""FFDNet plug-in denoiser adapter with online fine-tuning (``ffdnet_rgb_denoise_full_tensor``).

Mirror of packages/ffdnet/test_ffdnet_ipol.py:240-359: same name, arguments, layouts and return
convention.  The reference loops over the B frames calling ``model(img[1,3,H,W], sigma[1,1,1,1])``;
here the whole cube is one batch through the native conv engine, the Bayer sampling, the sensing
operator and the MSE of the measurement-consistency loss are one fused kernel that also emits the
gradient, backward runs on the native dgrad/wgrad kernels and Adam is one launch over the flat
parameter bucket (fresh optimizer state per call, like the reference's ``torch.optim.Adam`` at :251).
"""
import torch

from . import ops
from ._lib import SciError, call, ptr, stream
from .network_ffdnet import FFDNet

last_losses = []      # loss values of the most recent fine-tune call (the reference prints them, :298-299,:333-334)


def _unwrap(model):
    m = model.module if hasattr(model, "module") and not isinstance(model, FFDNet) else model
    if not isinstance(m, FFDNet):
        raise SciError("ffdnet adapter expects adaptivepnp_sci_b200.network_ffdnet.FFDNet, got %s" % type(m).__name__)
    return m


def _tile_loss(eng, out_ext, phi, y, dbuf_name, loss_slot, tile, want_grad):
    """Measurement loss (+ gradient) of a network output.  Tiled mode: the loss lives on this rank's own rows of the
    halo-extended strip and is normalised by the pixel count of the whole frame."""
    B = out_ext.shape[0]
    dev = out_ext.device
    if tile is None:
        H, W = out_ext.shape[2:]
        d = eng.ws.get(dbuf_name, tuple(out_ext.shape), dev) if want_grad else None
        call("sci_meas_loss_fwd_bwd", ptr(out_ext), ptr(phi), ptr(y), ptr(d), ptr(loss_slot), H, W, B, out_ext.shape[1], 0,
             stream())
        return d
    top, rows, W = tile.top, tile.rows, out_ext.shape[3]
    own = out_ext[:, :, top:top + rows].contiguous()
    d_own = eng.ws.get(dbuf_name + "_own", tuple(own.shape), dev) if want_grad else None
    call("sci_meas_loss_fwd_bwd", ptr(own), ptr(phi), ptr(y), ptr(d_own), ptr(loss_slot), rows, W, B, own.shape[1],
         tile.total_pixels, stream())
    if not want_grad:
        return None
    d = eng.ws.get(dbuf_name, tuple(out_ext.shape), dev)
    d.zero_()
    d[:, :, top:top + rows].copy_(d_own)
    return d


def finetune_and_denoise(u, phi, y, sigma, model, lr, update_per_iter, grad_sync=None, tile=None):
    """u [B,3,H,W], phi [B,H,W], y [H,W] planar.  update_per_iter Adam steps, then the eval forward.
    ``tile`` (parallel.TileView): u is a halo-extended row strip, phi / y cover this rank's own rows."""
    eng = _unwrap(model).engine()
    B, _, H, W = u.shape
    dev = u.device
    eng.prepare(training=True)
    eng.bucket.new_optimizer()
    loss = torch.zeros(update_per_iter + 1, dtype=torch.float64, device=dev)
    for it in range(update_per_iter):
        xhat = eng.forward(u, sigma, train=True)                                        # :266-273
        dxhat = _tile_loss(eng, xhat, phi, y, "dxhat", loss[it:it + 1], tile, True)     # :275-291
        eng.backward(dxhat)                                                             # :293
        if grad_sync is not None:
            grad_sync(eng.bucket.grad)
        eng.bucket.adam_step(lr)                                                        # :294
        eng.after_step()
    out = eng.forward(u, sigma, train=False)                                            # :303-315 (model.eval())
    _tile_loss(eng, out, phi, y, "dxhat", loss[update_per_iter:], tile, False)
    last_losses[:] = [loss]          # device tensor; read lazily by whoever wants to print it
    return out


def denoise_planar(u, pb, sigma, model, lr, do_update, update_per_iter, grad_sync=None, tile=None):
    """Solver-facing entry: planar in, planar out (a view of an engine buffer, consumed before the next call)."""
    if model is None:
        raise SciError("model_denoise is required")
    if do_update:
        return finetune_and_denoise(u, pb.phi, pb.y, sigma, model, lr, update_per_iter, grad_sync, tile)
    return _unwrap(model).engine().forward(u, sigma, train=False)


def ffdnet_rgb_denoise_full_tensor(x, yall, Phiall, sigma, model, useGPU=True, lr_=0.000001, updata_=False,
                                   update_per_iter=4, device=0):
    """x [H,W,3,B] CUDA, yall [h,w,4], Phiall [h,w,B,4], sigma float -> outv [H,W,3,B]
    (or ``(outv, model)`` when ``updata_``), exactly the reference's convention (:356-359).

    Reproducibility: the fine-tune's backward reductions (weight gradients, bias / BatchNorm column sums) run in a fixed
    order, so the same inputs, the same numpy / torch seeds (``utilspy.worker_init_fn``), the same GPU model and the same
    world size and transport give bit-identical outputs and bit-identical fine-tuned weights.  Not covered: NCCL's
    all-reduce in ``grad_sync`` (its algorithm choice; gloo is deterministic), DDnet's self-supervised update (never
    run by the solvers), and the printed fp64 diagnostics (PSNR, SSIM, losses), which may vary at ~1e-16 relative."""
    from .utils_image import fourCh2OneCh
    x = x.contiguous().float()
    H, W, _, B = x.shape
    u = ops.pixlast_to_planar(x, 3, B).view(B, 3, H, W)
    if updata_:
        phi = ops.pixlast_to_planar(fourCh2OneCh(Phiall.contiguous().float()), 1, B).view(B, H, W)
        y = fourCh2OneCh(yall.contiguous().float())
        out = finetune_and_denoise(u, phi, y, sigma, model, lr_, update_per_iter)
        vals = last_losses[0].cpu().numpy()
        for v in vals:
            print('loss:', end=' ')
            print('tensor(%.4e)' % v)
    else:
        out = _unwrap(model).engine().forward(u, sigma, train=False)
    outv = ops.planar_to_pixlast(out, 3, B).view(H, W, 3, B)
    return (outv, model) if updata_ else outv


def ffdnet_vdenoiser(vnoisy, sigma, model=None, useGPU=True):
    """packages/ffdnet/test_ffdnet_ipol.py:103-181 - frame-wise gray adapter: numpy ``vnoisy`` [M,N,F...] -> float64 numpy
    of the same shape, every frame ``frame - model(frame, sigma)`` without clipping (:177) with the IPOL-flavour gray model
    (``ffdnet_ipol_models.FFDNet(1)``, which returns the noise estimate).  The reference feeds the frames one by one; they
    are independent, so here the F frames are one batch through the native engine.  Like the reference (no odd-size
    handling, :146-158 commented out) it needs even M and N.  Not on the solvers' path; API parity (SURVEY 8(f).3)."""
    import numpy as np
    from .ffdnet_ipol_models import FFDNet as FFDNetIPOL
    if model is None:
        raise SciError("ffdnet_vdenoiser: pass the gray model (the reference's default models/net_gray.pth is not shipped, "
                       ".MISSING_LARGE_BLOBS)")
    if not useGPU:
        raise SciError("the native engine is CUDA only")
    net = model.module if hasattr(model, "module") and not isinstance(model, FFDNetIPOL) else model
    if not isinstance(net, FFDNetIPOL) or net.num_input_channels != 1:
        raise SciError("ffdnet_vdenoiser expects adaptivepnp_sci_b200.ffdnet_ipol_models.FFDNet(num_input_channels=1)")
    model.eval()                                                                          # :128
    vshape = vnoisy.shape
    v = np.ascontiguousarray(vnoisy, dtype=np.float32).reshape(vshape[0], vshape[1], -1)  # :132-133
    frames = torch.from_numpy(v).cuda().permute(2, 0, 1).unsqueeze(1).contiguous()        # [F,1,M,N]
    est = net.engine().forward(frames, float(sigma), train=False)
    out = (frames - est)[:, 0].permute(1, 2, 0).contiguous()                              # :177, no clamp
    return out.cpu().numpy().astype(np.float64).reshape(vshape)                           # outv is np.zeros(...): float64
