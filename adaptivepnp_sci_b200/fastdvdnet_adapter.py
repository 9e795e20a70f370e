"""FastDVDnet plug-in denoiser adapter with online fine-tuning.

Mirror of packages/fastdvdnet/test_fastdvdnet.py:325-500 (``fastdvdnet_denoiser_full_tensor_v2``) and
packages/fastdvdnet/fastdvdnet.py:82-146 (``fastdvdnet_seqdenoise``): same names, arguments, layouts,
return convention, and the same requirement that ``model`` exposes ``.module`` (the script wraps it in
``nn.DataParallel``, two_stage_ADMM_Online_FastDVD_Warm.py:240-241; ``DataParallelLike`` is the
single-device stand-in).

Fine-tune semantics reproduced from the reference:
* training input  vplus = v + float32(float64(v) + N(0,(5/255)^2))  — the helper at
  utils/utils_image.py:183-192 returns ``meas + noise`` and :359 adds ``vnoisy`` again — with the noise
  drawn on the HOST from the global numpy RNG (same call, same shape, same order), uploaded as float64;
* BatchNorm layers frozen in eval mode, but their affine parameters are trained (:376-385);
* fresh Adam state per (lr, n_iter) pair (:385); loss = MSE(sum_t Bayer(out_t)*Phi_t, y) over H*W (:428-431);
* final denoise of the CLEAN input with the updated weights (:453-458).
"""
import os

import numpy as np
import torch
import torch.nn as nn

from . import ops
from ._lib import SciError, call, ptr, stream
from .fastdvdnet_models import FastDVDnet

NUM_IN_FR_EXT = 5          # test_fastdvdnet.py:23
last_losses = []
_inflight = []             # (event, host noise array) pairs whose upload may still be running


class DataParallelLike(nn.Module):
    """Single-device stand-in for the ``nn.DataParallel`` wrapper of the script: ``.module`` attribute and
    ``module.``-prefixed state-dict keys (so a DataParallel checkpoint loads), no scatter/gather (every
    forward on the path is batch 1 in the reference, so DataParallel never split anything)."""

    def __init__(self, module, device_ids=None):
        super().__init__()
        self.module = module

    def forward(self, *a, **k):
        return self.module(*a, **k)


def _unwrap(model):
    m = model.module if hasattr(model, "module") else model
    if not isinstance(m, FastDVDnet):
        raise SciError("fastdvdnet adapter expects adaptivepnp_sci_b200.fastdvdnet_models.FastDVDnet, got %s"
                       % type(m).__name__)
    return m


def draw_finetune_noise(shape):
    """The reference's host-side draw (utils/utils_image.py:186): float64 N(0, 5/255) from the global numpy RNG."""
    return np.random.normal(0, 5 / 255, tuple(shape))


def fast_legacy_normal(rs, loc, scale, shape, nthreads=None):
    """``rs.normal(loc, scale, shape)`` for a legacy ``np.random.RandomState``, bit for bit (values and final state),
    computed by the multi-threaded host routine ``sci_host_legacy_normal`` (~5x faster than numpy on 16 cores)."""
    import ctypes
    from ._lib import lib
    name, key, pos, has_gauss, gauss = rs.get_state()
    if name != 'MT19937':
        return rs.normal(loc, scale, shape)
    key = np.ascontiguousarray(key, dtype=np.uint32).copy()
    n = int(np.prod(shape))
    out = _host_buffer(n)
    c_pos, c_has, c_g = ctypes.c_int(int(pos)), ctypes.c_int(int(has_gauss)), ctypes.c_double(float(gauss))
    rc = lib.sci_host_legacy_normal(key.ctypes.data_as(ctypes.c_void_p), ctypes.byref(c_pos), ctypes.byref(c_has),
                                    ctypes.byref(c_g), float(loc), float(scale), out.ctypes.data_as(ctypes.c_void_p), n,
                                    int(nthreads or _default_rng_threads()))
    if rc != 0:
        raise SciError("sci_host_legacy_normal failed (%d)" % rc)
    rs.set_state((name, key, c_pos.value, c_has.value, c_g.value))
    return out.reshape(shape)


def _default_rng_threads():
    """Worker threads of the host noise generator: the box's cores are shared by all ranks of the node (torchrun sets
    LOCAL_WORLD_SIZE), and the main thread of every rank must keep launching kernels while the helper draws ahead."""
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    ranks = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", os.environ.get("WORLD_SIZE", "1"))))
    return max(1, min(8, cores // ranks - 1))       # the Mersenne-Twister word stream is serial: 4-8 workers already hide the rest


_pool_lock = __import__("threading").Lock()
_pool = {}       # element count -> free page-locked float64 tensors
_owner = {}      # data pointer of a handed-out array -> the page-locked tensor that owns it


def _host_buffer(n):
    """float64 host array for the noise.  On a GPU box it lives in PINNED memory, so the upload in
    ``finetune_and_denoise`` is one asynchronous DMA instead of a staged, blocking pageable copy (2 x 50 MB per
    reconstruction at 512x512x8).  The buffers are pooled explicitly: page-locking 50 MB costs tens of milliseconds and
    takes driver locks that stall kernel launches, so after ``prewarm_host_buffers`` no allocation happens in steady state.
    (Whole-frame draws of the tiled mode are gigabytes per rank: page-locking those costs more than it saves.)"""
    if n <= (1 << 25) and torch.cuda.is_available() and os.environ.get("SCI_NOISE_PINNED", "1") != "0":
        with _pool_lock:
            free = _pool.get(n)
            t = free.pop() if free else None
        if t is None:
            try:
                t = torch.empty(n, dtype=torch.float64, pin_memory=True)
            except RuntimeError:
                t = None
        if t is not None:
            a = t.numpy()
            with _pool_lock:
                _owner[a.ctypes.data] = t
            return a
    return np.empty(n, dtype=np.float64)


def _release_host_buffer(arr):
    """Give a pooled buffer back once nothing reads it any more (no-op for ordinary numpy arrays)."""
    with _pool_lock:
        t = _owner.pop(arr.ctypes.data, None)
        if t is not None:
            _pool.setdefault(t.numel(), []).append(t)


def prewarm_host_buffers(n, count):
    """Page-lock ``count`` buffers of ``n`` doubles up front (first reconstruction), so later calls only recycle."""
    if not (n <= (1 << 25) and torch.cuda.is_available() and os.environ.get("SCI_NOISE_PINNED", "1") != "0"):
        return
    with _pool_lock:
        have = len(_pool.get(n, ()))
    fresh = []
    for _ in range(max(0, count - have)):
        try:
            fresh.append(torch.empty(n, dtype=torch.float64, pin_memory=True))
        except RuntimeError:
            break
    with _pool_lock:
        _pool.setdefault(n, []).extend(fresh)


def _state_key(st):
    """Comparable fingerprint of a numpy legacy RNG state tuple (MT19937 key, position, cached gaussian)."""
    return (st[0], st[1].tobytes(), st[2], st[3], st[4])


class NoiseStream:
    """Run-ahead producer of the fine-tune noise with EXACT global-RNG semantics.

    The reference draws ``np.random.normal(0, 5/255, [B,3,H,W])`` from the global numpy RNG inside every fine-tune
    call (~25 ns/sample on the legacy generator: 0.16 s for 8x3x512x512, comparable to the GPU time of a whole
    reconstruction).  A helper thread owns a PRIVATE ``RandomState`` cloned from the global state and keeps a few
    arrays ahead, remembering for each one the generator state before and after the draw.  ``get(shape)`` hands out
    the head array only if the global RNG is still exactly in that array's "before" state — i.e. nobody reseeded or
    drew anything else — and then moves the global RNG to the "after" state, which is precisely what the reference's
    call would have done.  Otherwise the queue is discarded, the array is drawn synchronously from the global RNG
    (again exactly like the reference) and the helper restarts from the new state.  Values and RNG state are
    therefore always identical to the reference's; only the wall-clock position of the work changes."""

    def __init__(self, depth=3):
        import threading
        self.depth = depth
        self.lock = threading.Condition()
        self.queue = []            # entries: (shape, key_before, state_after, array)
        self.shape = None
        self.rs = None             # private generator, positioned after the last queued array
        self.epoch = 0
        self.thread = None
        self.enabled = os.environ.get("SCI_NOISE_RUNAHEAD", "1") != "0"

    def _worker(self, epoch):
        while True:
            with self.lock:
                # whole-frame draws of the tiled mode are gigabytes each: keep one ahead, not ``depth``
                depth = 1 if int(np.prod(self.shape)) > (1 << 25) else self.depth
                while self.epoch == epoch and len(self.queue) >= depth:
                    self.lock.wait()
                if self.epoch != epoch:
                    return
                shape, rs = self.shape, self.rs
            before = _state_key(rs.get_state())
            arr = fast_legacy_normal(rs, 0, 5 / 255, shape)   # == rs.normal(0, 5/255, shape) (utils_image.py:186), bit for bit
            after = rs.get_state()
            with self.lock:
                if self.epoch != epoch:
                    _release_host_buffer(arr)         # drawn for a stream that was restarted meanwhile: back to the pool
                    return
                self.queue.append((shape, before, after, arr))
                self.lock.notify_all()

    def _restart(self, shape):
        """(Re)start the helper from the CURRENT global state; caller holds the lock."""
        import threading
        self.epoch += 1
        for _, _, _, arr in self.queue:
            _release_host_buffer(arr)
        self.queue = []
        if tuple(shape) != self.shape:
            prewarm_host_buffers(int(np.prod(shape)), self.depth + 3)
        self.shape = tuple(shape)
        self.rs = np.random.RandomState()
        self.rs.set_state(np.random.get_state())
        self.lock.notify_all()
        self.thread = threading.Thread(target=self._worker, args=(self.epoch,), daemon=True)
        self.thread.start()

    def prefetch(self, shape):
        """Hint that arrays of ``shape`` will be requested soon (called at the start of a reconstruction)."""
        if not self.enabled:
            return
        with self.lock:
            now = _state_key(np.random.get_state())
            ok = self.shape == tuple(shape) and ((self.queue and self.queue[0][1] == now) or
                                                 (not self.queue and self.rs is not None and
                                                  _state_key(self.rs.get_state()) == now))
            if not ok:
                self._restart(shape)

    def get(self, shape):
        shape = tuple(shape)
        if not self.enabled:
            return draw_finetune_noise(shape)
        with self.lock:
            now = _state_key(np.random.get_state())
            if self.shape == shape and self.thread is not None:
                # wait for the head if the helper is (about to be) producing the array that matches `now`
                while not self.queue and self.rs is not None and self.thread.is_alive():
                    self.lock.wait(timeout=0.05)
                    if self.queue:
                        break
                if self.queue and self.queue[0][0] == shape and self.queue[0][1] == now:
                    _, _, after, arr = self.queue.pop(0)
                    np.random.set_state(after)
                    self.lock.notify_all()
                    return arr
            # global RNG was reseeded / used elsewhere, or the shape changed: draw exactly like the reference
            arr = draw_finetune_noise(shape)
            self._restart(shape)
            return arr


noise_stream = NoiseStream()


def finetune_and_denoise(v, phi, y, sigma, model, lr, update_per_iter, grad_sync=None, noise=None, tile=None):
    """v [B,C,H,W], phi [B,H,W], y [H,W] planar; returns the denoised CLEAN sequence [B,C,H,W].  C = 3 with the colour
    model (Bayer measurement), C = 1 with the gray one (the measurement sums the frames themselves; the noise is drawn with
    shape (B,1,H,W); the twin that is trained is written back into the gray parameters after the last Adam step).
    ``tile`` (parallel.TileView): v is a halo-extended row strip of a larger frame, phi / y cover the own rows; the
    noise is drawn for the WHOLE frame (same global-RNG stream on every rank) and the strip's rows are cut out."""
    from .ffdnet_adapter import _tile_loss
    net = _unwrap(model)
    if v.shape[1] != net.num_color_channels:
        raise SciError("sequence has %d planes, the model %d" % (v.shape[1], net.num_color_channels))
    eng = net.engine()
    B, C, H, W = v.shape
    dev = v.device
    if isinstance(update_per_iter, int):
        n_update_iter, lr_all = [update_per_iter], [lr]                                  # :344-349
    else:
        n_update_iter, lr_all = list(update_per_iter), list(lr)
    full = None
    if noise is None:
        if tile is None:
            noise = noise_stream.get((B, C, H, W))
        else:
            full = noise_stream.get((B, C, tile.H_total, W))
            noise = full[:, :, tile.g0:tile.g0 + H]
    noise_h = np.ascontiguousarray(noise, dtype=np.float64)
    if full is not None and noise_h.ctypes.data != full.ctypes.data:
        _release_host_buffer(full)           # the strip was copied out: the whole-frame buffer is free again
    noise_d = torch.from_numpy(noise_h).to(dev, non_blocking=True)        # pinned source -> one asynchronous DMA
    # the host buffer must outlive the DMA (the host runs ahead of the stream): park it until its event has fired
    ev = torch.cuda.Event()
    ev.record()
    still = []
    for e, a in _inflight:
        if e.query():
            _release_host_buffer(a)          # its upload has completed: the pinned buffer goes back to the pool
        else:
            still.append((e, a))
    _inflight[:] = still + [(ev, noise_h)]
    vplus = eng.ws.get("vplus", (B, C, H, W), dev)
    call("sci_fastdvd_noisy_input", ptr(v), ptr(noise_d), ptr(vplus), v.numel(), stream())    # :359
    eng.prepare(training=True)
    n_steps = int(sum(n_update_iter))
    loss = torch.zeros(n_steps + 1, dtype=torch.float64, device=dev)
    k = 0
    for lr_i, nit in zip(lr_all, n_update_iter):
        eng.bucket.new_optimizer()                                                        # :385
        for _ in range(nit):
            out = eng.forward(vplus, sigma, train=True)                                   # :412-419
            dout = _tile_loss(eng, out, phi, y, "dout", loss[k:k + 1], tile, True)        # :428-431
            eng.backward(dout)                                                            # :445
            if grad_sync is not None:
                grad_sync(eng.bucket.grad)
            eng.bucket.adam_step(lr_i)                                                    # :446
            eng.after_step()
            k += 1
    if net.num_color_channels == 1:
        net._restrict_twin()
    out = eng.forward(v, sigma, train=False)                                              # :453-458
    _tile_loss(eng, out, phi, y, "dout", loss[n_steps:], tile, False)
    last_losses[:] = [loss]
    return out


def denoise_planar(u, pb, sigma, model, lr, do_update, update_per_iter, grad_sync=None, noise=None, tile=None):
    """Solver-facing entry: planar in, planar out (engine buffer, consumed before the next call)."""
    if model is None:
        raise SciError("model_denoise is required")
    if do_update:
        return finetune_and_denoise(u, pb.phi, pb.y, sigma, model, lr, update_per_iter, grad_sync, noise, tile)
    return _unwrap(model).engine().forward(u, sigma, train=False)


def fastdvdnet_seqdenoise(seq, noise_std, windsize, model, train=None):
    """fastdvdnet.py:82-146 — seq [N,C,H,W] -> [N,C,H,W], circular 5-frame window (C = 3, or 1 with the gray model, whose
    frames the engine packs as the first plane of a colour cube: fastdvdnet_models.FastDVDnet)."""
    if windsize != NUM_IN_FR_EXT:
        raise NotImplementedError("window size 5 only")
    net = _unwrap(model)
    if seq.shape[1] != net.num_color_channels:
        raise SciError("sequence has %d channels, the model %d" % (seq.shape[1], net.num_color_channels))
    seq = seq.contiguous().float()
    padded, H, W = ops.pad_to_multiple(seq, 4)                                          # reflect pad to x4 (:119-127)
    out = net.engine().forward(padded, float(noise_std.flatten()[0]), train=False)
    out = ops.crop_to(out, H, W).clone()                                                # un-pad (:134-141)
    return (out, model) if train else out


def fastdvdnet_denoiser_full_tensor_v2(vnoisy, sigma, y_bayer=None, Phi=None, model=None,
                                       useGPU=True, lr_=0.000001, updata_=False, update_per_iter=1, gray=False,
                                       update_times=-1):
    """vnoisy [H,W,3,B] CUDA, y_bayer [h,w,4], Phi [h,w,B,4] -> outv [H,W,3,B] (or ``(outv, model)``).

    Reproducibility: the fine-tune's backward reductions (weight gradients, bias / BatchNorm column sums) run in a fixed
    order, so the same inputs, the same numpy / torch seeds (``utilspy.worker_init_fn``), the same GPU model and the same
    world size and transport give bit-identical outputs and bit-identical fine-tuned weights.  Not covered: NCCL's
    all-reduce in ``grad_sync`` (its algorithm choice; gloo is deterministic), DDnet's self-supervised update (never
    run by the solvers), and the printed fp64 diagnostics (PSNR, SSIM, losses), which may vary at ~1e-16 relative."""
    from .utils_image import fourCh2OneCh
    if gray:
        raise NotImplementedError("the full-tensor adapter serves the Bayer solvers (colour cube [H,W,3,B]); the gray model "
                                  "runs through the frame-wise fastdvdnet_denoiser(gray=True)")
    vnoisy = vnoisy.contiguous().float()
    H, W, _, B = vnoisy.shape
    v = ops.pixlast_to_planar(vnoisy, 3, B).view(B, 3, H, W)
    if updata_:
        _ = model.module                                                                   # :377 requires the wrapper
        phi = ops.pixlast_to_planar(fourCh2OneCh(Phi.contiguous().float()), 1, B).view(B, H, W)
        y = fourCh2OneCh(y_bayer.contiguous().float())
        out = finetune_and_denoise(v, phi, y, sigma, model, lr_, update_per_iter)
        for val in last_losses[0].cpu().numpy():
            print('loss:', end=' ')
            print('tensor(%.4e)' % val)
    else:
        out = _unwrap(model).engine().forward(v, sigma, train=False)
    outv = ops.planar_to_pixlast(out, 3, B).view(H, W, 3, B)
    return (outv, model) if updata_ else outv


def fastdvdnet_denoiser(vnoisy, sigma, model=None, useGPU=True, lr_=0.000001, updata_=False, gray=False):
    """packages/fastdvdnet/test_fastdvdnet.py:149-235 - frame-wise adapter: numpy ``vnoisy`` [H,W,F,3] (``gray=True``:
    [H,W,F], with the single-channel model ``FastDVDnet(num_color_channels=1)``) in [0,1] -> numpy of the same shape, the
    whole circular sequence through ``fastdvdnet_seqdenoise``.

    Not on the hot path (the solvers call ``fastdvdnet_denoiser_full_tensor_v2``); kept for API parity (SURVEY 8(f).3).
    ``updata_=True`` takes one Adam step on MSE(input, output) - a self-loss no script uses and whose backward is not
    built here; it raises."""
    if updata_:
        raise NotImplementedError("fastdvdnet_denoiser(updata_=True) (MSE(input, output) self-loss) is not on any script's path; "
                                  "the online adaptation of the solvers is fastdvdnet_denoiser_full_tensor_v2")
    if model is None:
        raise SciError("model is required")
    v = torch.from_numpy(np.ascontiguousarray(vnoisy, dtype=np.float32)).cuda()           # [H,W,F,3] / [H,W,F]
    if gray:
        v = v.unsqueeze(3)                                                                  # :212-213
    seq = v.permute(2, 3, 0, 1).contiguous()                                                # :215 -> [F,C,H,W]
    out = fastdvdnet_seqdenoise(seq, torch.tensor([float(sigma)], device=seq.device), NUM_IN_FR_EXT, model)
    out = out.permute(2, 3, 0, 1)                                                           # :226
    if gray:
        out = out.squeeze(3)                                                                # :227-228
    return out.contiguous().cpu().numpy()
