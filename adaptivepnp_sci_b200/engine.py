"""Native execution engine of the two denoisers (forward, backward, Adam) on the sm_100a kernels.

The networks of the reference are short, fixed chains of 3x3 convolutions; this module is
the host-side schedule that strings the C-ABI kernels together:

* activations: NHWC fp32, channels padded to a multiple of 32 (padded channels hold zeros);
* weights: PyTorch parameters (fp32 master copies, one flat bucket per model so that Adam
  and the NCCL gradient all-reduce are single launches) re-packed into the implicit-GEMM
  layout ``[9][Cout][Cin]`` whenever they change; BatchNorm (always in eval mode on this
  path, test_fastdvdnet.py:376-379) is folded into the per-column scale/shift epilogue;
* forward  = ``sci_conv3x3_fwd`` per layer (bias/BN + ReLU + skip-add + PixelShuffle fused);
* backward = ``sci_act_bwd`` -> ``sci_conv3x3_wgrad`` -> ``sci_conv3x3_dgrad`` per layer, the
  measurement loss and its gradient in one kernel (``sci_meas_loss_fwd_bwd``), one fused
  ``sci_adam_step`` over the flat bucket.

``SCI_CONV_IMPL`` selects the convolution kernels: ``tc`` (default; tcgen05/TMEM/TMA, TF32
operands, fp32 accumulation) or ``ref`` (fp32 FFMA on-device reference).  Both are CUDA;
there is no PyTorch/CPU path.
"""
import ctypes
import os

import torch
import torch.nn as nn

from . import _lib
from ._lib import call, ptr, stream

_f32p = ctypes.c_void_p


class ConvDesc(ctypes.Structure):
    _fields_ = [("x", _f32p), ("w", _f32p), ("scale", _f32p), ("shift", _f32p), ("residual", _f32p), ("y", _f32p),
                ("N", ctypes.c_int), ("H", ctypes.c_int), ("W", ctypes.c_int), ("Cin", ctypes.c_int),
                ("Cout", ctypes.c_int), ("stride", ctypes.c_int), ("relu", ctypes.c_int),
                ("pixel_shuffle", ctypes.c_int), ("round_tf32", ctypes.c_int), ("w_split", ctypes.c_int), ("emit_lo", ctypes.c_int),
                ("planar_in1", _f32p), ("planar_out", _f32p), ("pdl", ctypes.c_int),
                ("half_io", ctypes.c_int), ("Cin_store", ctypes.c_int), ("Cout_store", ctypes.c_int),
                ("mask_y", _f32p), ("col_s1", _f32p), ("col_s2", _f32p), ("mask_relu", ctypes.c_int), ("lo_channel0", ctypes.c_int),
                ("K_used", ctypes.c_int), ("planar_planes", ctypes.c_int), ("workspace", ctypes.c_void_p),
                ("workspace_bytes", ctypes.c_size_t)]


class WgradDesc(ctypes.Structure):
    _fields_ = [("x", _f32p), ("dz", _f32p), ("oscale", _f32p), ("dw", _f32p),
                ("N", ctypes.c_int), ("H", ctypes.c_int), ("W", ctypes.c_int), ("Cin", ctypes.c_int),
                ("Cout", ctypes.c_int), ("stride", ctypes.c_int), ("workspace", ctypes.c_void_p),
                ("workspace_bytes", ctypes.c_size_t)]


class LayerOp(ctypes.Structure):
    """sci_layer_op (include/sci_b200.h): one entry of a batched bookkeeping launch."""
    _fields_ = [("kind", ctypes.c_int), ("Co", ctypes.c_int), ("Ci", ctypes.c_int), ("groups", ctypes.c_int),
                ("Co_pad", ctypes.c_int), ("Ci_pad", ctypes.c_int), ("ps", ctypes.c_int), ("tflip", ctypes.c_int),
                ("round_tf32", ctypes.c_int), ("ci_dup", ctypes.c_int), ("eps", ctypes.c_float),
                ("a", _f32p), ("b", _f32p), ("c", _f32p), ("d", _f32p), ("o0", _f32p), ("o1", _f32p)]

    def elements(self):
        k = self.kind
        if k in (0, 2):
            return 9 * self.Co_pad * self.Ci_pad
        if k == 1:
            return 9 * 4 * self.Ci_pad * self.Co_pad
        if k == 3:
            return self.Co * (self.Ci // self.groups) * 9
        return self.Co_pad if k == 4 else self.Co


def _op(kind, Co=0, Ci=1, groups=1, Co_pad=0, Ci_pad=0, ps=0, tflip=0, round_tf32=0, ci_dup=0, eps=0.0, a=None, b=None, c=None,
        d=None, o0=None, o1=None):
    return LayerOp(kind, Co, Ci, groups, Co_pad, Ci_pad, int(ps), int(tflip), int(round_tf32), ci_dup, eps,
                   _dp(a), _dp(b), _dp(c), _dp(d), _dp(o0), _dp(o1))


class OpTable:
    """Device-resident table of LayerOps run as ONE launch (``sci_layer_ops_batch``)."""

    def __init__(self, ops, device):
        self.n = len(ops)
        arr = (LayerOp * self.n)(*ops)
        self.dev = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).to(device)
        self.max_blocks = max((op.elements() + 255) // 256 for op in ops)

    def run(self):
        call("sci_layer_ops_batch", ptr(self.dev), self.n, self.max_blocks, stream())


IMPL_TC, IMPL_REF = 0, 1


def default_impl():
    v = os.environ.get("SCI_CONV_IMPL", "tc").lower()
    if v not in ("tc", "ref"):
        raise ValueError("SCI_CONV_IMPL must be 'tc' or 'ref'")
    return IMPL_TC if v == "tc" else IMPL_REF


def _pad(c, m):
    return (c + m - 1) // m * m


def _dp(t):
    return None if t is None else t.data_ptr()


class ParamBucket:
    """All trainable parameters of a model as views of ONE flat fp32 CUDA buffer (+ flat grad, Adam moments)."""

    def __init__(self, params):
        self.params = [p for p in params if p.requires_grad]
        if not self.params:
            raise _lib.SciError("model has no trainable parameters")
        dev = self.params[0].device
        if dev.type != "cuda":
            raise _lib.SciError("move the model to the GPU before using it (model.cuda())")
        self.sizes = [p.numel() for p in self.params]
        self.offsets = [0]
        for n in self.sizes:
            self.offsets.append(self.offsets[-1] + _pad(n, 4))          # 16-byte aligned slots
        self.total = self.offsets[-1]
        self.flat = torch.zeros(self.total, dtype=torch.float32, device=dev)
        self.grad = torch.zeros(self.total, dtype=torch.float32, device=dev)
        self.exp_avg = None
        self.exp_avg_sq = None
        self.step = 0
        for p, off, n in zip(self.params, self.offsets, self.sizes):
            view = self.flat[off:off + n].view(p.shape)
            view.copy_(p.data)
            p.data = view

    def intact(self):
        base = self.flat.data_ptr()
        return all(p.data_ptr() == base + 4 * off for p, off in zip(self.params, self.offsets))

    def grad_view(self, p):
        i = next(k for k, q in enumerate(self.params) if q is p)
        return self.grad[self.offsets[i]:self.offsets[i] + self.sizes[i]].view(p.shape)

    def new_optimizer(self):
        """Fresh Adam state, as the reference re-creates the optimizer on every adapter call."""
        if self.exp_avg is None:
            self.exp_avg = torch.zeros_like(self.flat)
            self.exp_avg_sq = torch.zeros_like(self.flat)
        else:
            self.exp_avg.zero_()
            self.exp_avg_sq.zero_()
        self.step = 0

    def adam_step(self, lr, betas=(0.9, 0.999), eps=1e-8):
        self.step += 1
        call("sci_adam_step", ptr(self.flat), ptr(self.grad), ptr(self.exp_avg), ptr(self.exp_avg_sq), self.total,
             float(lr), float(betas[0]), float(betas[1]), float(eps), self.step, stream())


class ConvLayer:
    """One 3x3 convolution of a network with its epilogue and its packed device-side state."""

    def __init__(self, conv, bn=None, relu=False, stride=1, ps=False, cin_pad=None, first=False, wsplit=False,
                 dup_in=False):
        self.conv, self.bn, self.relu, self.stride, self.ps = conv, bn, relu, stride, ps
        self.Co, self.groups = conv.out_channels, conv.groups
        self.Ci = conv.in_channels
        self.Ci_pad = cin_pad or _pad(self.Ci, 32)
        self.dup_in = dup_in     # input tensor carries [hi | remainder] halves of Ci_pad channels each (emit_lo producer)
        if dup_in:
            self.ci_half = self.Ci_pad
            self.Ci_pad *= 2
        # multiple of 32: it is the K extent of the data-gradient GEMM.  PixelShuffle layers: four sub-pixel groups of
        # pad(Co/4, 32) columns each, so that the up-sampled tensor is itself 32-channel padded
        self.Co_pad = 4 * _pad(self.Co // 4, 32) if ps else _pad(self.Co, 32)
        self.out_ch = self.Co_pad // 4 if ps else self.Co_pad       # channels of the stored output tensor
        dev = conv.weight.device
        self.wsplit = wsplit     # TF32 path: keep tf32(w) AND the remainder tf32(w - tf32(w)); both are multiplied
        self.wpk = torch.empty((18 if wsplit else 9) * self.Co_pad * self.Ci_pad, dtype=torch.float32, device=dev)
        self.wpk_t = None
        self.has_affine = bn is not None or conv.bias is not None
        self.scale = torch.empty(self.Co_pad, dtype=torch.float32, device=dev) if bn is not None else None
        self.shift = torch.zeros(self.Co_pad, dtype=torch.float32, device=dev) if self.has_affine else None
        self.s1 = self.s2 = None
        self.dwpk = None
        self.first = first       # network input layer: on the TF32 path its input arrives as hi + remainder copies

    # ---- table entries of the engine's batched bookkeeping launches (one launch per phase, see _EngineBase._table) ----
    def fwd_ops(self, tf32):
        c = self.conv
        ops = []
        if self.bn is not None:
            bn = self.bn
            ops.append(_op(4, Co=self.Co, Co_pad=self.Co_pad, eps=float(bn.eps), a=bn.weight.data, b=bn.bias.data,
                           c=bn.running_mean, d=bn.running_var, o0=self.scale, o1=self.shift))
        elif c.bias is not None:
            ops.append(_op(6, Co=self.Co, a=c.bias.data, o0=self.shift))
        self.ci_dup = self.ci_half if self.dup_in else (16 if (self.first and tf32) else 0)
        ops.append(_op(0, self.Co, self.Ci, self.groups, self.Co_pad, self.Ci_pad, self.ps, 0,
                       (2 if (tf32 and self.wsplit) else int(tf32)), self.ci_dup, a=c.weight.data, o0=self.wpk))
        return ops

    def bwd_ops(self, tf32, s1, s2):
        """Allocates the data-gradient weights; s1 / s2 are this layer's slices of the engine's flat column-sum buffer."""
        dev = self.wpk.device
        self.s1, self.s2 = s1, s2
        self.s2t = bool(self.stride == 2 and self.groups == 1 and not self.ps and self.ci_dup == 0)
        n = (36 if self.s2t else 9) * self.Co_pad * self.Ci_pad
        if self.wpk_t is None or self.wpk_t.numel() != n:
            self.wpk_t = torch.empty(n, dtype=torch.float32, device=dev)
        if self.s2t:
            return [_op(1, Co=self.Co, Ci=self.Ci, Co_pad=self.Co_pad, Ci_pad=self.Ci_pad, round_tf32=int(tf32),
                        a=self.conv.weight.data, b=self.scale, o0=self.wpk_t)]
        return [_op(0, self.Co, self.Ci, self.groups, self.Co_pad, self.Ci_pad, self.ps, 1, int(tf32), self.ci_dup,
                    a=self.conv.weight.data, b=self.scale, o0=self.wpk_t)]

    def grad_ops(self, bucket):
        ops = [_op(3, self.Co, self.Ci, self.groups, self.Co_pad, self.Ci_pad, self.ps, ci_dup=self.ci_dup, a=self.dwpk,
                   o0=bucket.grad_view(self.conv.weight))]
        if self.bn is not None:
            ops.append(_op(5, Co=self.Co, a=self.s1, b=self.s2, c=self.bn.weight.data, d=self.bn.bias.data,
                           o0=bucket.grad_view(self.bn.weight), o1=bucket.grad_view(self.bn.bias)))
        elif self.conv.bias is not None:
            ops.append(_op(6, Co=self.Co, a=self.s1, o0=bucket.grad_view(self.conv.bias)))
        return ops


class HalfLayer:
    """fp16 forward form of a ConvLayer (inference chains on the kind::f16 kernels, ``sci_conv_desc.half_io``).

    Shares the fp32 layer's epilogue vectors (folded BatchNorm scale / shift: same GEMM column layout); its own state is the
    packed fp16 weight tensor ``[9][N][K]`` with ``N = Co_pad`` GEMM columns and ``K`` = stored input channels rounded up to
    64 (one 128-byte operand row).  ``cin_store`` / ``cout_store`` are the channels per pixel of the fp16 NHWC tensors it
    reads / writes (96 for the 90-channel tensor, otherwise 64 or 128; tensors with 32 real channels carry 32 zeros)."""

    def __init__(self, base, cin_store, cout_store, ci_dup=0, split=False):
        self.base = base
        self.cin_store, self.cout_store, self.ci_dup = cin_store, cout_store, ci_dup
        self.split = split
        if split:
            # value + remainder form (sci_conv_desc.w_split with half_io): a 64-channel chunk per 32 real channels on the
            # input, the weights and the output; ci_dup = -1 selects that weight layout
            self.ci_dup = -1
            self.cin_store = 2 * _pad(base.Ci, 32)
            self.cout_store = 2 * base.Co_pad
        self.K = 32 if self.cin_store == 32 else _pad(self.cin_store, 64)   # 32-channel tensors: 64-byte operand rows (SWIZZLE_64B)
        self.k_used = (ci_dup + base.Ci) if ci_dup else base.Ci        # leading K columns that can be non-zero
        self.N = base.Co_pad
        self.stride, self.relu, self.ps = base.stride, base.relu, base.ps
        self.wpk = torch.empty(9 * self.N * self.K, dtype=torch.float16, device=base.conv.weight.device)

    def fwd_ops(self, tf32):
        b = self.base
        return [_op(2, b.Co, b.Ci, b.groups, self.N, self.K, self.ps, ci_dup=self.ci_dup, a=b.conv.weight.data, o0=self.wpk)]


class _Workspace:
    """Named, shape-keyed device buffers that live as long as the engine (no allocation in steady state)."""

    def __init__(self):
        self.bufs = {}

    def get(self, name, shape, device, zero=False, dtype=torch.float32):
        key = (name, tuple(shape), dtype)
        t = self.bufs.get(key)
        if t is None:
            t = torch.empty(shape, dtype=dtype, device=device)
            self.bufs[key] = t
            if zero:
                t.zero_()
        elif zero:
            t.zero_()
        return t


class _EngineBase:
    def __init__(self, module, layers):
        self.module = module
        self.layers = layers
        self.impl = default_impl()
        self.tf32 = self.impl == IMPL_TC
        self.ws = _Workspace()
        self.bucket = None
        self._seen_version = None
        self._bwd_valid = False
        self.dirty = True
        self.n_launch = 0
        self._tables = None
        self.s12_flat = None
        self.pdl_chain = False   # True inside an inference chain: weights are packed, consecutive convs may overlap (PDL)
        self.red_buf = None      # scratch of the fixed-order reductions of the backward pass (grown on demand, see _red_ws)
        self.profile = None      # set to a list to record (start_event, end_event, algorithmic_flops, tag) per conv launch

    # ---- parameter state ------------------------------------------------------------------------------
    def _version(self):
        v = 0
        for t in list(self.module.parameters()) + list(self.module.buffers()):
            v += t._version
        return v

    def prepare(self, training=False):
        """Make the packed device-side state consistent with the module's parameters."""
        if self.bucket is None or not self.bucket.intact():
            self.bucket = ParamBucket(list(self.module.parameters()))
            self.dirty = True
        if self._tables is not None and self._tables["bucket"] is not self.bucket:
            self._tables = None                                       # new parameter storage: every table entry points at the old one
        if self.dirty or self._version() != self._seen_version:
            self._table("fwd").run()
            self._seen_version = self._version()
            self._bwd_valid = False
            self.dirty = False
        if training and self.layers[0].dwpk is None:
            sizes = [9 * L.Co_pad * L.Ci_pad for L in self.layers]
            self.dw_flat = torch.zeros(sum(sizes), dtype=torch.float32, device=self.layers[0].wpk.device)
            off = 0
            for L, n in zip(self.layers, sizes):
                L.dwpk = self.dw_flat[off:off + n]
                off += n
        if training and not self._bwd_valid:
            self._table("bwd").run()
            self._bwd_valid = True

    def _table(self, which):
        """Batched bookkeeping, one launch per phase: 'fwd' = BatchNorm folding / bias + weight
        packing of every layer (+ the fp16 / split inference forms), 'bwd' = data-gradient weight forms, 'grads' = packed
        weight gradients -> parameter gradients + BatchNorm / bias gradients from the column sums."""
        if self._tables is None:
            self._tables = {"bucket": self.bucket}
        t = self._tables.get(which)
        if t is None:
            dev = self.layers[0].wpk.device
            if which == "fwd":
                ops = [op for L in self.layers + (getattr(self, "layers_inf", None) or []) for op in L.fwd_ops(self.tf32)]
            elif which == "bwd":
                if self.s12_flat is None:
                    self.s12_flat = torch.zeros(2 * sum(L.Co_pad for L in self.layers), dtype=torch.float32, device=dev)
                ops, off = [], 0
                for L in self.layers:
                    ops += L.bwd_ops(self.tf32, self.s12_flat[off:off + L.Co_pad], self.s12_flat[off + L.Co_pad:off + 2 * L.Co_pad])
                    off += 2 * L.Co_pad
            else:
                ops = [op for L in self.layers for op in L.grad_ops(self.bucket)]
            t = self._tables[which] = OpTable(ops, dev)
        return t

    def begin_backward(self):
        """Zero the packed weight-gradient accumulators and the per-column sums (one memset each)."""
        self.dw_flat.zero_()
        self.s12_flat.zero_()

    def param_grads(self, L):
        """Per-layer step of the parameter gradients of L: nothing is left to do per layer, finish_param_grads() computes
        those of every layer in one launch.  Kept so that callers which drive a backward pass layer by layer still work."""

    def finish_param_grads(self):
        """All parameter gradients in one launch at the end of the backward pass: packed dW -> torch-layout grad slots,
        bias / BatchNorm affine grads from the column sums."""
        self._table("grads").run()
        self.n_launch += 1

    def _red_ws(self, nbytes, device):
        """Scratch for the fixed-order (bit-reproducible) reductions of one backward call: each CTA stores its partial
        weight gradient / column sums into its own slot, a second kernel adds the slots in slot order.  One buffer serves
        every call of the stream in turn; it grows to the largest need seen (the widest layer's slots, 29 MB for the
        128->128 FastDVDnet layers at 8x512x512), so nothing is allocated in steady state."""
        if self.red_buf is None or self.red_buf.numel() < nbytes:
            self.red_buf = torch.empty(nbytes, dtype=torch.uint8, device=device)
        return self.red_buf.data_ptr()

    def _ordered(self, d, query, dev):
        """Give descriptor d (ConvDesc / WgradDesc) the reduction workspace its call needs (none: left NULL)."""
        need = getattr(_lib.lib, query)(ctypes.byref(d), self.impl)
        if need:
            d.workspace = self._red_ws(need, dev)
            d.workspace_bytes = need

    # ---- kernel wrappers ------------------------------------------------------------------------------
    def conv(self, L, x, N, H, W, y, residual=None, round_out=True, emit_lo=False, planar=None):
        """planar = (in1, out) planar [N,P,H,W] tensors (P = 3, or 1 for gray frames): tensor-core path only, fused
        `out = in1 - conv` (y unused)."""
        d = ConvDesc(_dp(x), _dp(L.wpk), _dp(L.scale), _dp(L.shift), _dp(residual), _dp(y), N, H, W, L.Ci_pad, L.Co_pad,
                     L.stride, int(L.relu), int(L.ps), int(self.tf32 and round_out), int(self.tf32 and L.wsplit),
                     int(emit_lo), _dp(planar[0]) if planar else None, _dp(planar[1]) if planar else None,
                     int(self.pdl_chain))
        if L.dup_in and self.tf32 and L.wsplit:
            d.lo_channel0 = L.ci_half                # "3xTF32": the remainder half of the input starts here (split accumulators)
        if planar:
            d.planar_planes = planar[0].shape[1]
        if self.profile is not None:
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
        call("sci_conv3x3_fwd", ctypes.byref(d), self.impl, stream())
        if self.profile is not None:
            ev1.record()
            Ho, Wo = (H - 1) // L.stride + 1, (W - 1) // L.stride + 1
            self.profile.append((ev0, ev1, 2.0 * N * Ho * Wo * 9 * (L.Ci // L.groups) * L.Co,
                                 "fwd %dx%d %d->%d s%d" % (H, W, L.Ci, L.Co, L.stride)))
        self.n_launch += 1

    def conv_h(self, Lh, x, N, H, W, y, residual=None, planar=None):
        """fp16 inference conv (tensor-core path only): x / y / residual are torch.float16 NHWC tensors."""
        b = Lh.base
        d = ConvDesc(_dp(x), _dp(Lh.wpk), _dp(b.scale), _dp(b.shift), _dp(residual), _dp(y), N, H, W, Lh.K, Lh.N,
                     Lh.stride, int(Lh.relu), int(Lh.ps), 0, int(Lh.split), 0, _dp(planar[0]) if planar else None,
                     _dp(planar[1]) if planar else None, int(self.pdl_chain), 1, Lh.cin_store, Lh.cout_store)
        d.K_used = Lh.k_used                         # zero-padded channels of the last 64-channel chunk are not multiplied
        if planar:
            d.planar_planes = planar[0].shape[1]
        if self.profile is not None:
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
        call("sci_conv3x3_fwd", ctypes.byref(d), IMPL_TC, stream())
        if self.profile is not None:
            ev1.record()
            Ho, Wo = (H - 1) // Lh.stride + 1, (W - 1) // Lh.stride + 1
            self.profile.append((ev0, ev1, 2.0 * N * Ho * Wo * 9 * (b.Ci // b.groups) * b.Co,
                                 "fwd %dx%d %d->%d s%d" % (H, W, b.Ci, b.Co, Lh.stride)))
        self.n_launch += 1

    def _mask_args(self, d, mask):
        """mask = (y_prev, L_prev): fuse the activation backward of the layer that produced this dgrad's output tensor."""
        if mask is not None:
            y_prev, Lp = mask
            d.mask_y = _dp(y_prev)
            d.col_s1 = _dp(Lp.s1) if Lp.has_affine else None
            d.col_s2 = _dp(Lp.s2) if Lp.bn is not None else None
            d.mask_relu = int(Lp.relu)

    def can_fuse_act_bwd(self, Lp, out_channels):
        """The data-gradient kernel can apply layer Lp's activation backward in its epilogue (tensor-core fp32 path)."""
        return self.impl == IMPL_TC and (Lp.relu or Lp.has_affine) and out_channels <= 128

    def dgrad_s2(self, L, dz, N, Ho, Wo, dx, residual=None, mask=None):
        """Stride-2 layer: dx[N,2Ho,2Wo,Ci_pad] = PixelShuffle(conv(dz[N,Ho,Wo,Co_pad], sub-pixel weights)) [+ residual]."""
        d = ConvDesc(_dp(dz), _dp(L.wpk_t), None, None, _dp(residual), _dp(dx), N, Ho, Wo, L.Co_pad, 4 * L.Ci_pad, 1, 0, 1,
                     int(self.tf32), 0, 0)
        self._mask_args(d, mask)
        if mask is not None:
            self._ordered(d, "sci_conv3x3_fwd_workspace_bytes", dz.device)
        call("sci_conv3x3_dgrad", ctypes.byref(d), self.impl, stream())
        self.n_launch += 1

    def dgrad(self, L, dz, N, Ho, Wo, dx, residual=None, mask=None):
        """dx[N,Ho,Wo,Ci_pad] = conv(dz, packed transposed+flipped (and BN-scaled) weights) [+ residual]."""
        d = ConvDesc(_dp(dz), _dp(L.wpk_t), None, None, _dp(residual), _dp(dx), N, Ho, Wo, L.Co_pad, L.Ci_pad, 1, 0, 0,
                     int(self.tf32), 0, 0)
        self._mask_args(d, mask)
        if mask is not None:
            self._ordered(d, "sci_conv3x3_fwd_workspace_bytes", dz.device)
        call("sci_conv3x3_dgrad", ctypes.byref(d), self.impl, stream())
        self.n_launch += 1

    def wgrad(self, L, x, dz, N, H, W):
        """L.dwpk += packed weight gradient, reduced over the CTAs in a fixed order (bit-identical on every run)."""
        d = WgradDesc(_dp(x), _dp(dz), _dp(L.scale), _dp(L.dwpk), N, H, W, L.Ci_pad, L.Co_pad, L.stride)
        self._ordered(d, "sci_conv3x3_wgrad_workspace_bytes", dz.device)
        call("sci_conv3x3_wgrad", ctypes.byref(d), self.impl, stream())
        self.n_launch += 2

    def act_bwd(self, L, dy, y, n_pix, C):
        """dz (in place over dy) = dy * relu'(y); accumulates the per-column sums needed for bias / BN grads (fixed order)."""
        need = L.has_affine
        if not (L.relu or need):
            return dy
        yp = ptr(y) if (L.relu or L.bn is not None) else None
        if not need:
            call("sci_act_bwd", ptr(dy), yp, ptr(dy), n_pix, C, int(L.relu), None, None, stream())
            self.n_launch += 1
            return dy
        nb = _lib.lib.sci_act_bwd_workspace_bytes(n_pix, C)
        call("sci_act_bwd_ordered", ptr(dy), yp, ptr(dy), n_pix, C, int(L.relu), ptr(L.s1),
             ptr(L.s2) if L.bn is not None else None, self._red_ws(nb, dy.device), nb, stream())
        self.n_launch += 2
        return dy

    def after_step(self):
        """Parameters were updated in place by sci_adam_step (raw pointers): re-pack on next use."""
        self.dirty = True


class FFDNetEngine(_EngineBase):
    """models/network_ffdnet.py:54-69 on the native kernels, all frames of a cube as one batch."""

    def __init__(self, module):
        # conv_layers(): convolutions in execution order, each a Conv2d or a (Conv2d, BatchNorm2d) pair (the IPOL flavour,
        # ffdnet_ipol_models.py, has inference-mode BatchNorm between its inner layers)
        convs = [c if isinstance(c, tuple) else (c, None) for c in module.conv_layers()]
        layers = []
        for i, (c, bn) in enumerate(convs):
            last = i == len(convs) - 1
            # FFDNet returns the denoised image itself (no residual), so weight-rounding error reaches the output
            # undamped: on the TF32 path its weights are kept as tf32 hi + remainder (north_star 1e-3 max-abs bound).
            # This also holds for the TRAINING forward: with plain TF32 weights there (1.75 ms instead of 3.5 ms per pass at
            # 8x512x512, tools/time_ffdnet_train.py) the Adam-normalised updates change enough to move the final
            # reconstruction by 5e-3 on the golden online loop (3.4e-4 with the split), so the split stays on.
            layers.append(ConvLayer(c, bn, relu=not last, first=(i == 0), wsplit=default_impl() == IMPL_TC))
        super().__init__(module, layers)
        # inference on the TF32 path keeps every activation and weight as a value + remainder pair, which brings the conv
        # stack to ~fp32 accuracy (FFDNet has no residual connection, so plain TF32 rounding reaches the output undamped
        # and is then integrated by the ADMM dual variables): as fp16 value + fp16 remainder (x 2^11) on the row-reuse
        # kernel, three products at the fp16 tensor rate and half the bytes ...
        self.layers_h = None
        if self.tf32 and os.environ.get("SCI_FFDNET_INF", "half") == "half" and all(L.Co_pad <= 128 for L in layers):
            self.layers_h = [HalfLayer(L, 0, 0, split=True) for L in layers]
        # ... or, with SCI_FFDNET_INF=tf32 or a layer wider than 128 columns, as "3xTF32": tf32 hi + remainder
        self.layers_inf = self.layers_h                  # (the list prepare() re-packs)
        if self.tf32 and self.layers_h is None:
            self.layers_inf = [ConvLayer(c, bn, relu=(i < len(convs) - 1), first=(i == 0), wsplit=True, dup_in=(i > 0))
                               for i, (c, bn) in enumerate(convs)]
        self.in_nc, self.out_nc = module.in_nc, module.out_nc
        if (self.in_nc, self.out_nc) not in ((3, 3), (1, 1)):
            raise NotImplementedError("native FFDNet engine: colour (3->3) and gray (1->1) models")

    def forward(self, u, sigma, train=False):
        """u [B,C,H,W] planar fp32 (C = 3 colour / 1 gray) -> xhat [B,C,H,W].  train=True keeps the activations."""
        B, _, H, W = u.shape
        if H % 2 or W % 2:
            raise _lib.SciError("native FFDNet engine needs even H and W (Bayer frames always are)")
        self.prepare(training=train)
        dev = u.device
        h2, w2 = H // 2, W // 2
        if not train and self.layers_h is not None:
            return self._forward_split_half(u, sigma, B, H, W)
        if not train and self.layers_inf is not None:
            return self._forward_precise(u, sigma, B, H, W)
        L0 = self.layers[0]
        a = self.ws.get("in", (B, h2, w2, L0.Ci_pad), dev)
        call("sci_ffdnet_pack_input", ptr(u), float(sigma), ptr(a), B, self.in_nc, H, W, L0.Ci_pad, int(self.tf32), stream())
        acts = [a]
        for i, L in enumerate(self.layers):
            name = ("act%d" % i) if train else ("pp%d" % (i % 2) if i < len(self.layers) - 1 else "tail")
            y = self.ws.get(name, (B, h2, w2, L.Co_pad), dev)
            self.conv(L, acts[-1], B, h2, w2, y, round_out=i < len(self.layers) - 1)
            acts.append(y)
        xhat = self.ws.get("xhat_train" if train else "xhat", (B, self.out_nc, H, W), dev)
        call("sci_ffdnet_unpack_output", ptr(acts[-1]), ptr(xhat), B, self.out_nc, H, W, self.layers[-1].Co_pad, stream())
        if train:
            self._saved = (acts, B, H, W)
        return xhat

    def _forward_split_half(self, u, sigma, B, H, W):
        dev = u.device
        h2, w2 = H // 2, W // 2
        a = self.ws.get("in_h", (B, h2, w2, 64), dev, dtype=torch.float16)
        call("sci_ffdnet_pack_input_split_half", ptr(u), float(sigma), ptr(a), B, self.in_nc, H, W, stream())
        self.n_launch += 1
        for i, Lh in enumerate(self.layers_h):
            y = self.ws.get("hpp%d" % (i % 2), (B, h2, w2, Lh.cout_store), dev, dtype=torch.float16)
            self.conv_h(Lh, a, B, h2, w2, y)
            a = y
        xhat = self.ws.get("xhat", (B, self.out_nc, H, W), dev)
        call("sci_ffdnet_unpack_output_split_half", ptr(a), ptr(xhat), B, self.out_nc, H, W, stream())
        self.n_launch += 1
        return xhat

    def _forward_precise(self, u, sigma, B, H, W):
        dev = u.device
        h2, w2 = H // 2, W // 2
        Ls = self.layers_inf
        a = self.ws.get("in", (B, h2, w2, Ls[0].Ci_pad), dev)
        call("sci_ffdnet_pack_input", ptr(u), float(sigma), ptr(a), B, self.in_nc, H, W, Ls[0].Ci_pad, 1, stream())
        for i, L in enumerate(Ls):
            last = i == len(Ls) - 1
            y = self.ws.get("tail" if last else "ppx%d" % (i % 2), (B, h2, w2, L.Co_pad * (1 if last else 2)), dev)
            self.conv(L, a, B, h2, w2, y, round_out=not last, emit_lo=not last)
            a = y
        xhat = self.ws.get("xhat", (B, self.out_nc, H, W), dev)
        call("sci_ffdnet_unpack_output", ptr(a), ptr(xhat), B, self.out_nc, H, W, Ls[-1].Co_pad, stream())
        return xhat

    def backward(self, dxhat):
        """Gradients of all parameters into the flat grad bucket, given d(loss)/d(xhat) [B,3,H,W]."""
        acts, B, H, W = self._saved
        dev = dxhat.device
        h2, w2 = H // 2, W // 2
        n_pix = B * h2 * w2
        self.begin_backward()
        Lt = self.layers[-1]
        dy = self.ws.get("g_tail", (B, h2, w2, Lt.Co_pad), dev)
        call("sci_ffdnet_unpack_output_grad", ptr(dxhat), ptr(dy), B, self.out_nc, H, W, Lt.Co_pad, stream())
        for i in range(len(self.layers) - 1, -1, -1):
            L = self.layers[i]
            dz = self.act_bwd(L, dy, acts[i + 1], n_pix, L.Co_pad)
            self.wgrad(L, acts[i], dz, B, h2, w2)
            if i > 0:
                dx = self.ws.get("g%d" % (i % 2), (B, h2, w2, L.Ci_pad), dev)
                self.dgrad(L, dz, B, h2, w2, dx)
                dy = dx
        self.finish_param_grads()

    def forward_nchw(self, x, sigma):
        """Reference call convention model(img[N,3,H,W], sigma[N,1,1,1]) (test_ffdnet_ipol.py:350-351)."""
        from . import ops
        s = float(sigma.flatten()[0])
        if sigma.numel() > 1 and not bool((sigma == sigma.flatten()[0]).all()):
            raise NotImplementedError("one noise level per call on the native path")
        # odd sizes: replication pad to even, crop the result (network_ffdnet.py:56-59, :68)
        xp, H, W = ops.replicate_pad_to_even(x.contiguous().float())
        return ops.crop_to(self.forward(xp, s, train=False), H, W).clone()


class _DenBlockLayers:
    """The 16 convolutions of one DenBlock (packages/fastdvdnet/models.py:146-198) as ConvLayers."""

    def __init__(self, block):
        specs = block.conv_specs()
        self.L = []
        for i, (conv, bn, relu, stride, ps) in enumerate(specs):
            self.L.append(ConvLayer(conv, bn, relu=relu, stride=stride, ps=ps, first=(i == 0)))


class FastDVDnetEngine(_EngineBase):
    """packages/fastdvdnet/models.py:200-253 + the circular sequence driver fastdvdnet.py:82-146, with every
    temp1 triple evaluated once (B distinct triples instead of 3B; identical values, SURVEY App. C)."""

    # stored channels per pixel of each layer's fp16 input / output tensor (see HalfLayer): the 90-channel tensor keeps 96,
    # 32-channel tensors are stored as 64 (32 zeros) so that every pixel row is one 128-byte operand row
    _H_IN = [64, 96, 64, 64, 64, 64, 128, 128, 128, 128, 128, 64, 64, 64, 64, 64]
    _H_OUT = [96, 64, 64, 64, 64, 128, 128, 128, 128, 128, 64, 64, 64, 64, 64, 64]
    # since the 64-byte-row (SWIZZLE_64B) kernels: tensors with 32 real channels (packed input, x0, s0, o0) are stored as 32
    _H_IN32 = [32, 96, 32, 64, 64, 64, 128, 128, 128, 128, 128, 64, 64, 64, 32, 32]
    _H_OUT32 = [96, 32, 64, 64, 64, 128, 128, 128, 128, 128, 64, 64, 64, 32, 32, 32]

    def __init__(self, module):
        self.t1 = _DenBlockLayers(module.temp1)
        self.t2 = _DenBlockLayers(module.temp2)
        super().__init__(module, self.t1.L + self.t2.L)
        # inference chains in fp16 (kind::f16 MMAs, fp32 accumulation: TF32's 11-bit significand, half the bytes, twice the
        # tensor rate); SCI_CONV_HALF=0 keeps them on the TF32 kernels
        self.half = self.impl == IMPL_TC and os.environ.get("SCI_CONV_HALF", "1") != "0"
        self.layers_inf = None
        if self.half:
            self.sw64 = os.environ.get("SCI_CONV_SW64", "1") != "0"
            hin, hout = (self._H_IN32, self._H_OUT32) if self.sw64 else (self._H_IN, self._H_OUT)
            self.t1h = [HalfLayer(L, ci, co, ci_dup=16 if i == 0 else 0) for i, (L, ci, co) in enumerate(zip(self.t1.L, hin, hout))]
            self.t2h = [HalfLayer(L, ci, co, ci_dup=16 if i == 0 else 0) for i, (L, ci, co) in enumerate(zip(self.t2.L, hin, hout))]
            self.layers_inf = self.t1h + self.t2h

    def _block_forward_h(self, Lh, frames, sigma, out):
        """One DenBlock on the fp16 kernels (inference): planar fp32 frames in, planar fp32 ``frames - net`` out."""
        B, C, H, W = frames.shape
        dev = frames.device
        f16 = torch.float16
        g = lambda n, shape: self.ws.get("h_" + n, shape, dev, dtype=f16)
        h2, w2, h4, w4 = H // 2, W // 2, H // 4, W // 4
        c32 = Lh[0].cin_store                # 32 (64-byte pixel rows) or 64: channels per pixel of the 32-channel tensors
        a_in = g("in", (B, H, W, c32))
        call("sci_fastdvd_pack_input_half_planes", ptr(frames), float(sigma), ptr(a_in), B, C, H, W, c32, stream())
        a0 = g("a0", (B, H, W, 96));        self.conv_h(Lh[0], a_in, B, H, W, a0)
        x0 = g("x0", (B, H, W, c32));       self.conv_h(Lh[1], a0, B, H, W, x0)
        d0a = g("d0a", (B, h2, w2, 64));    self.conv_h(Lh[2], x0, B, H, W, d0a)
        d0b = g("d0b", (B, h2, w2, 64));    self.conv_h(Lh[3], d0a, B, h2, w2, d0b)
        x1 = g("x1", (B, h2, w2, 64));      self.conv_h(Lh[4], d0b, B, h2, w2, x1)
        d1a = g("d1a", (B, h4, w4, 128));   self.conv_h(Lh[5], x1, B, h2, w2, d1a)
        d1b = g("d1b", (B, h4, w4, 128));   self.conv_h(Lh[6], d1a, B, h4, w4, d1b)
        x2 = g("x2", (B, h4, w4, 128));     self.conv_h(Lh[7], d1b, B, h4, w4, x2)
        u2a = g("u2a", (B, h4, w4, 128));   self.conv_h(Lh[8], x2, B, h4, w4, u2a)
        u2b = g("u2b", (B, h4, w4, 128));   self.conv_h(Lh[9], u2a, B, h4, w4, u2b)
        s1 = g("s1", (B, h2, w2, 64));      self.conv_h(Lh[10], u2b, B, h4, w4, s1, residual=x1)
        u1a = g("u1a", (B, h2, w2, 64));    self.conv_h(Lh[11], s1, B, h2, w2, u1a)
        u1b = g("u1b", (B, h2, w2, 64));    self.conv_h(Lh[12], u1a, B, h2, w2, u1b)
        s0 = a_in                           # the packed input is dead once a0 exists; x0 once s0 exists
        self.conv_h(Lh[13], u1b, B, h2, w2, s0, residual=x0)
        o0 = x0
        self.conv_h(Lh[14], s0, B, H, W, o0)
        self.conv_h(Lh[15], o0, B, H, W, None, planar=(frames, out))

    # ---- one DenBlock ---------------------------------------------------------------------------------
    def _block_forward(self, tag, blk, frames, sigma, out, train):
        B, C, H, W = frames.shape
        dev = frames.device
        L = blk.L
        g = self.ws.get
        keep = (lambda n: "%s_%s" % (tag, n)) if train else (lambda n: "inf_" + n)
        h2, w2, h4, w4 = H // 2, W // 2, H // 4, W // 4
        a_in = g(keep("in"), (B, H, W, L[0].Ci_pad), dev)
        call("sci_fastdvd_pack_input_planes", ptr(frames), float(sigma), ptr(a_in), B, C, H, W, L[0].Ci_pad, int(self.tf32),
             stream())
        a0 = g(keep("a0"), (B, H, W, L[0].Co_pad), dev);   self.conv(L[0], a_in, B, H, W, a0)
        x0 = g(keep("x0"), (B, H, W, L[1].Co_pad), dev);   self.conv(L[1], a0, B, H, W, x0)
        d0a = g(keep("d0a"), (B, h2, w2, 64), dev);        self.conv(L[2], x0, B, H, W, d0a)
        d0b = g(keep("d0b"), (B, h2, w2, 64), dev);        self.conv(L[3], d0a, B, h2, w2, d0b)
        x1 = g(keep("x1"), (B, h2, w2, 64), dev);          self.conv(L[4], d0b, B, h2, w2, x1)
        d1a = g(keep("d1a"), (B, h4, w4, 128), dev);       self.conv(L[5], x1, B, h2, w2, d1a)
        d1b = g(keep("d1b"), (B, h4, w4, 128), dev);       self.conv(L[6], d1a, B, h4, w4, d1b)
        x2 = g(keep("x2"), (B, h4, w4, 128), dev);         self.conv(L[7], d1b, B, h4, w4, x2)
        u2a = g(keep("u2a"), (B, h4, w4, 128), dev);       self.conv(L[8], x2, B, h4, w4, u2a)
        u2b = g(keep("u2b"), (B, h4, w4, 128), dev);       self.conv(L[9], u2a, B, h4, w4, u2b)
        s1 = g(keep("s1"), (B, h2, w2, 64), dev);          self.conv(L[10], u2b, B, h4, w4, s1, residual=x1)
        u1a = g(keep("u1a"), (B, h2, w2, 64), dev);        self.conv(L[11], s1, B, h2, w2, u1a)
        u1b = g(keep("u1b"), (B, h2, w2, 64), dev);        self.conv(L[12], u1a, B, h2, w2, u1b)
        # inference: the packed input is dead once a0 exists and x0 once s0 exists -> s0 / o0 reuse their buffers (two
        # full-resolution tensors less: 26 GB at 2048x2048x24)
        alias = (not train) and L[0].Ci_pad == 32 and L[1].Co_pad == 32
        s0 = a_in if alias else g(keep("s0"), (B, H, W, 32), dev)
        self.conv(L[13], u1b, B, h2, w2, s0, residual=x0)
        o0 = x0 if alias else g(keep("o0"), (B, H, W, 32), dev)
        self.conv(L[14], s0, B, H, W, o0)
        if self.impl == IMPL_TC and L[15].Co_pad == 32:
            xo = None                                       # fused epilogue: out = frames - conv, planar, no NHWC tensor
            self.conv(L[15], o0, B, H, W, None, round_out=False, planar=(frames, out))
        else:
            xo = g(keep("xo"), (B, H, W, L[15].Co_pad), dev);  self.conv(L[15], o0, B, H, W, xo, round_out=False)
            call("sci_fastdvd_output_planes", ptr(frames), ptr(xo), ptr(out), B, C, H, W, L[15].Co_pad, stream())
        if train:
            return dict(a_in=a_in, a0=a0, x0=x0, d0a=d0a, d0b=d0b, x1=x1, d1a=d1a, d1b=d1b, x2=x2, u2a=u2a, u2b=u2b,
                        s1=s1, u1a=u1a, u1b=u1b, s0=s0, o0=o0, xo=xo)
        return None

    def forward(self, frames, sigma, train=False):
        """frames [B,C,H,W] planar -> denoised [B,C,H,W] (whole circular sequence).  C = 3, or C = 1: gray frames on the
        colour-shaped embedding of the gray model (fastdvdnet_models.FastDVDnet), which the boundary kernels pack as the
        first plane of a colour cube whose other planes are zero, and of whose output only the first plane is computed."""
        B, C, H, W = frames.shape
        if C not in (1, 3):
            raise _lib.SciError("native FastDVDnet engine: frames with 3 (colour) or 1 (gray) planes, got %d" % C)
        if H % 4 or W % 4:
            raise NotImplementedError("native FastDVDnet engine needs H, W multiples of 4 (the reference reflect-pads, "
                                      "fastdvdnet.py:119-127; the hot-path sizes never need it)")
        self.prepare(training=train)
        dev = frames.device
        t1_out = self.ws.get("t1_out_train" if train else "t1_out", (B, C, H, W), dev)
        out = self.ws.get("out_train" if train else "out", (B, C, H, W), dev)
        # inference: the packed weights are final before the first conv starts, so consecutive layers may overlap their
        # prologue with the previous layer's tail (programmatic dependent launch); not while profiling per layer
        self.pdl_chain = (not train) and self.profile is None and self.impl == IMPL_TC
        try:
            if self.half and not train:
                self._block_forward_h(self.t1h, frames, sigma, t1_out)
                self._block_forward_h(self.t2h, t1_out, sigma, out)
                s1 = s2 = None
            else:
                s1 = self._block_forward("t1", self.t1, frames, sigma, t1_out, train)
                s2 = self._block_forward("t2", self.t2, t1_out, sigma, out, train)
        finally:
            self.pdl_chain = False
        if train:
            self._saved = (s1, s2, B, H, W)
        return out

    BLOCK_HALO = 40      # rows: one DenBlock sees -38..+36 full-resolution rows (two stride-2 levels, 16 convs); multiple of 4

    def forward_tiled(self, u_own, sigma, tile):
        """Inference on a row strip of a larger frame (``parallel.TileContext``): u_own [B,3,rows,W] -> denoised own rows.

        One halo exchange PER DenBlock (40 rows each) instead of one 80-row halo for the two-block cascade: block 1 runs on
        the strip extended by 40 rows, its own rows are exact; their boundary rows are exchanged again and block 2 runs on
        that.  Redundant convolution work: (rows + 80) / rows instead of (rows + 160) / rows (1.31 vs 1.62 at 256-row strips).
        Zero padding is only ever applied at true image borders, so the result equals the un-tiled one."""
        B, _, rows, W = u_own.shape
        self.prepare(training=False)
        dev = u_own.device
        h = self.BLOCK_HALO
        ext1, top = tile.exchange(u_own, h)
        t1_ext = self.ws.get("tl_t1", tuple(ext1.shape), dev)
        self.pdl_chain = self.profile is None and self.impl == IMPL_TC
        try:
            self._run_block(0, ext1, sigma, t1_ext)
            t1_own = t1_ext[:, :, top:top + rows].contiguous()
            ext2, top = tile.exchange(t1_own, h)
            out_ext = self.ws.get("tl_out", tuple(ext2.shape), dev)
            self._run_block(1, ext2, sigma, out_ext)
        finally:
            self.pdl_chain = False
        return out_ext[:, :, top:top + rows].contiguous()

    def _run_block(self, which, frames, sigma, out):
        if self.half:
            self._block_forward_h(self.t1h if which == 0 else self.t2h, frames, sigma, out)
        else:
            self._block_forward("t%d" % (which + 1), self.t1 if which == 0 else self.t2, frames, sigma, out, False)

    # ---- backward of one DenBlock -----------------------------------------------------------------------
    def _block_backward(self, blk, S, dout, B, H, W, need_input_grad):
        """dout [B,C,H,W] = d loss / d block output.  Returns d loss / d (packed input) [B,H,W,32] or None."""
        L = blk.L
        dev = dout.device
        g = self.ws.get
        h2, w2, h4, w4 = H // 2, W // 2, H // 4, W // 4
        nf, nh, nq = B * H * W, B * h2 * w2, B * h4 * w4

        Y = {0: "a0", 1: "x0", 2: "d0a", 3: "d0b", 4: "x1", 5: "d1a", 6: "d1b", 7: "x2", 8: "u2a", 9: "u2b", 11: "u1a", 12: "u1b", 14: "o0"}
        fused = set()        # layers whose dz was already produced by the data-gradient kernel of the layer after them

        def layer_bwd(i, dy, y, x_in, N, Hin, Win, n_out_pix, dx_name, dx_shape, residual=None, want_dx=True, prev=None):
            """Backward of layer i given dy wrt its stored output y; returns dx (grad wrt its input).  prev = index of the layer
            whose stored output IS this layer's input tensor: its activation backward is fused into this layer's data gradient
            (dx then already is that layer's dz)."""
            Li = L[i]
            dz = dy if i in fused else self.act_bwd(Li, dy, y, n_out_pix, Li.Co_pad)
            self.wgrad(Li, x_in, dz, N, Hin, Win)
            dx = None
            if want_dx:
                dx = g(dx_name, dx_shape, dev)
                mask = None
                if prev is not None and self.can_fuse_act_bwd(L[prev], dx_shape[-1]):
                    mask = (S[Y[prev]], L[prev])
                    fused.add(prev)
                if Li.stride == 2 and getattr(Li, "s2t", False):
                    self.dgrad_s2(Li, dz, N, Hin // 2, Win // 2, dx, residual, mask=mask)
                elif Li.stride == 2:
                    if mask is not None:
                        fused.discard(prev)
                    dil = g("g_dil", (N, Hin, Win, Li.Co_pad), dev)
                    call("sci_nhwc_dilate2", ptr(dz), ptr(dil), N, Hin // 2, Win // 2, Li.Co_pad, stream())
                    self.dgrad(Li, dil, N, Hin, Win, dx, residual)
                else:
                    Ho, Wo = Hin, Win
                    self.dgrad(Li, dz, N, Ho, Wo, dx, residual, mask=mask)
            return dx

        # out = in1 - xo  ->  d xo = -dout (padded columns 0)
        d_xo = g("g_xo", (B, H, W, L[15].Co_pad), dev)
        call("sci_fastdvd_output_grad_planes", ptr(dout), ptr(d_xo), B, dout.shape[1], H, W, L[15].Co_pad, stream())
        d_o0 = layer_bwd(15, d_xo, S["xo"], S["o0"], B, H, W, nf, "g_f32a", (B, H, W, 32), prev=14)
        d_s0 = layer_bwd(14, d_o0, S["o0"], S["s0"], B, H, W, nf, "g_f32b", (B, H, W, 32))
        # s0 = x0 + PS(conv13(u1b)): gradient of the GEMM output is the pixel-unshuffle of d_s0
        d_c13 = g("g_h128", (B, h2, w2, 128), dev)
        call("sci_nhwc_pixel_unshuffle", ptr(d_s0), ptr(d_c13), B, h2, w2, 32, stream())
        d_u1b = layer_bwd(13, d_c13, None, S["u1b"], B, h2, w2, nh, "g_h64a", (B, h2, w2, 64), prev=12)
        d_u1a = layer_bwd(12, d_u1b, S["u1b"], S["u1a"], B, h2, w2, nh, "g_h64b", (B, h2, w2, 64), prev=11)
        d_s1 = layer_bwd(11, d_u1a, S["u1a"], S["s1"], B, h2, w2, nh, "g_h64a", (B, h2, w2, 64))
        d_c10 = g("g_q256", (B, h4, w4, 256), dev)
        call("sci_nhwc_pixel_unshuffle", ptr(d_s1), ptr(d_c10), B, h4, w4, 64, stream())
        d_u2b = layer_bwd(10, d_c10, None, S["u2b"], B, h4, w4, nq, "g_q128a", (B, h4, w4, 128), prev=9)
        d_u2a = layer_bwd(9, d_u2b, S["u2b"], S["u2a"], B, h4, w4, nq, "g_q128b", (B, h4, w4, 128), prev=8)
        d_x2 = layer_bwd(8, d_u2a, S["u2a"], S["x2"], B, h4, w4, nq, "g_q128a", (B, h4, w4, 128), prev=7)
        d_d1b = layer_bwd(7, d_x2, S["x2"], S["d1b"], B, h4, w4, nq, "g_q128b", (B, h4, w4, 128), prev=6)
        d_d1a = layer_bwd(6, d_d1b, S["d1b"], S["d1a"], B, h4, w4, nq, "g_q128a", (B, h4, w4, 128), prev=5)
        # x1 feeds conv5 (stride 2) and the skip into s1: total gradient = dgrad + d_s1
        d_x1 = layer_bwd(5, d_d1a, S["d1a"], S["x1"], B, h2, w2, nq, "g_h64b", (B, h2, w2, 64), residual=d_s1, prev=4)
        d_d0b = layer_bwd(4, d_x1, S["x1"], S["d0b"], B, h2, w2, nh, "g_h64a", (B, h2, w2, 64), prev=3)
        d_d0a = layer_bwd(3, d_d0b, S["d0b"], S["d0a"], B, h2, w2, nh, "g_h64b", (B, h2, w2, 64), prev=2)
        d_x0 = layer_bwd(2, d_d0a, S["d0a"], S["x0"], B, H, W, nh, "g_f32a", (B, H, W, 32), residual=d_s0, prev=1)
        d_a0 = layer_bwd(1, d_x0, S["x0"], S["a0"], B, H, W, nf, "g_f96", (B, H, W, L[0].Co_pad), prev=0)
        return layer_bwd(0, d_a0, S["a0"], S["a_in"], B, H, W, nf, "g_fin", (B, H, W, L[0].Ci_pad),
                         want_dx=need_input_grad)

    def backward(self, dout):
        """Parameter gradients of both DenBlocks given d loss / d output [B,C,H,W]."""
        s1, s2, B, H, W = self._saved
        dev = dout.device
        self.begin_backward()
        d_in2 = self._block_backward(self.t2, s2, dout, B, H, W, need_input_grad=True)
        # temp1 output j feeds slot (j - f + 1) of temp2 block f = j-1, j, j+1, and is `in1` of block j
        C = dout.shape[1]
        d_t1 = self.ws.get("g_t1", (B, C, H, W), dev)
        d_t1.copy_(dout)
        call("sci_fastdvd_pack_input_grad_planes", ptr(d_in2), ptr(d_t1), B, C, H, W, self.t2.L[0].Ci_pad, 1, stream())
        self._block_backward(self.t1, s1, d_t1, B, H, W, need_input_grad=False)
        self.finish_param_grads()

    def forward_window(self, x, noise_map):
        """Reference call convention model(x[1,15,H,W], noise_map[1,1,H,W]) for ONE 5-frame window
        (packages/fastdvdnet/models.py:227-251); API parity only — the solvers use forward()."""
        if x.shape[0] != 1 or x.shape[1] != 15:
            raise _lib.SciError("expected x of shape [1,15,H,W]")
        sigma = float(noise_map.flatten()[0])
        frames = x.view(5, 3, x.shape[2], x.shape[3]).contiguous().float()
        B, _, H, W = frames.shape
        self.prepare(False)
        dev = frames.device
        t1 = self.ws.get("win_t1", (5, 3, H, W), dev)
        out = self.ws.get("win_out", (5, 3, H, W), dev)
        self._block_forward("w1", self.t1, frames, sigma, t1, False)      # centres 1,2,3 are the window's triples
        self._block_forward("w2", self.t2, t1, sigma, out, False)         # block 2 reads temp1 results 1,2,3
        return out[2:3].clone()


class DDnetEngine(_EngineBase):
    """models/network_demosaicking.py:377-463 + the circular sequence driver packages/DDnet/DDnet_test.py:166-204 on the
    native kernels (inference; the solvers never fine-tune the demosaicker, dvp:193,243 pass no ``args``).

    The three temp1 triples / three temp11 triples of all B centre frames run as ONE batch of 3B images each, the two
    temp2 evaluations as one batch of 2B.  Real channel widths 20/40/80/90 are zero-padded to 32/64/96/96."""

    def __init__(self, module):
        def body(block):
            return [ConvLayer(c, None, relu=r, stride=st, ps=ps, first=(i == 0))
                    for i, (c, r, st, ps) in enumerate(block.conv_specs())]
        self.t1, self.t11, self.t2 = body(module.temp1), body(module.temp11), body(module.temp2)
        self.fus = [ConvLayer(c, None, relu=r, stride=st, ps=ps, first=(i == 0))
                    for i, (c, r, st, ps) in enumerate(module.temp11.fusion_specs())]
        super().__init__(module, self.t1 + self.t11 + self.fus + self.t2)

    def _body(self, L, a_in, N, H, W, keep=None, cap=None):
        """The 16-conv U-shaped body shared by all DenBlock variants (:232-241): returns the last conv's output.
        ``keep`` (a tag): every activation gets its own buffer and the dict of them is returned too (training).
        ``cap`` >= N: buffers are allocated for ``cap`` images and used for the first N (the ragged last frame chunk)."""
        dev = a_in.device
        g = lambda name, shape, dev: self.ws.get(name, (cap or shape[0],) + shape[1:], dev)[:shape[0]]
        h2, w2, h4, w4 = H // 2, W // 2, H // 4, W // 4
        S = {"a_in": a_in}

        def run(i, x, n_h, n_w, name, residual=None, round_out=True):
            Li = L[i]
            ho, wo = (n_h // 2, n_w // 2) if Li.stride == 2 else ((n_h * 2, n_w * 2) if Li.ps else (n_h, n_w))
            y = g(("dd_%s_%s" % (keep, name)) if keep else ("dd_" + name), (N, ho, wo, Li.out_ch), dev)
            self.conv(Li, x, N, n_h, n_w, y, residual=residual, round_out=round_out)
            S[name] = y
            return y
        a0 = run(0, a_in, H, W, "a0")
        x0 = run(1, a0, H, W, "x0")
        d0a = run(2, x0, H, W, "d0a")
        d0b = run(3, d0a, h2, w2, "d0b")
        x1 = run(4, d0b, h2, w2, "x1")
        d1a = run(5, x1, h2, w2, "d1a")
        d1b = run(6, d1a, h4, w4, "d1b")
        x2 = run(7, d1b, h4, w4, "x2")
        u2a = run(8, x2, h4, w4, "u2a")
        u2b = run(9, u2a, h4, w4, "u2b")
        s1 = run(10, u2b, h4, w4, "s1", residual=x1)           # x1 + PixelShuffle(conv)
        u1a = run(11, s1, h2, w2, "u1a")
        u1b = run(12, u1a, h2, w2, "u1b")
        s0 = run(13, u1b, h2, w2, "s0", residual=x0)
        o0 = run(14, s0, H, W, "o0")
        xo = run(15, o0, H, W, "xo", round_out=False)
        return (xo, S) if keep else xo

    def _layer_bwd(self, Li, dy, y, x_in, N, Hin, Win, dx_name, residual=None, want_dx=True):
        """Backward of one conv layer given dy w.r.t. its stored output y: weight gradient, then dx (w.r.t. its input)."""
        dev = dy.device
        Ho, Wo = (Hin // 2, Win // 2) if Li.stride == 2 else (Hin, Win)
        dz = self.act_bwd(Li, dy, y, N * Ho * Wo, Li.Co_pad)
        self.wgrad(Li, x_in, dz, N, Hin, Win)
        dx = None
        if want_dx:
            dx = self.ws.get(dx_name, (N, Hin, Win, Li.Ci_pad), dev)
            if Li.stride == 2:
                self.dgrad_s2(Li, dz, N, Ho, Wo, dx, residual)
            else:
                self.dgrad(Li, dz, N, Ho, Wo, dx, residual)
        return dx

    def _body_backward(self, L, S, d_xo, N, H, W, want_dx, tag):
        """Adjoint of _body: parameter gradients of its 16 convs; returns d loss / d a_in (or None)."""
        dev = d_xo.device
        g = self.ws.get
        h2, w2, h4, w4 = H // 2, W // 2, H // 4, W // 4
        nm = lambda n: "ddg_%s_%s" % (tag, n)
        bw = self._layer_bwd
        d_o0 = bw(L[15], d_xo, None, S["o0"], N, H, W, nm("f_a"))
        d_s0 = bw(L[14], d_o0, S["o0"], S["s0"], N, H, W, nm("f_b"))
        # s0 = x0 + PixelShuffle(conv13(u1b)): the gradient of the GEMM output is the pixel-unshuffle of d_s0
        d_c13 = g(nm("c13"), (N, h2, w2, L[13].Co_pad), dev)
        call("sci_nhwc_pixel_unshuffle", ptr(d_s0), ptr(d_c13), N, h2, w2, L[13].out_ch, stream())
        d_u1b = bw(L[13], d_c13, None, S["u1b"], N, h2, w2, nm("h_a"))
        d_u1a = bw(L[12], d_u1b, S["u1b"], S["u1a"], N, h2, w2, nm("h_b"))
        d_s1 = bw(L[11], d_u1a, S["u1a"], S["s1"], N, h2, w2, nm("h_a"))
        d_c10 = g(nm("c10"), (N, h4, w4, L[10].Co_pad), dev)
        call("sci_nhwc_pixel_unshuffle", ptr(d_s1), ptr(d_c10), N, h4, w4, L[10].out_ch, stream())
        d_u2b = bw(L[10], d_c10, None, S["u2b"], N, h4, w4, nm("q_a"))
        d_u2a = bw(L[9], d_u2b, S["u2b"], S["u2a"], N, h4, w4, nm("q_b"))
        d_x2 = bw(L[8], d_u2a, S["u2a"], S["x2"], N, h4, w4, nm("q_a"))
        d_d1b = bw(L[7], d_x2, S["x2"], S["d1b"], N, h4, w4, nm("q_b"))
        d_d1a = bw(L[6], d_d1b, S["d1b"], S["d1a"], N, h4, w4, nm("q_a"))
        d_x1 = bw(L[5], d_d1a, S["d1a"], S["x1"], N, h2, w2, nm("h_b"), residual=d_s1)     # x1 also feeds the skip into s1
        d_d0b = bw(L[4], d_x1, S["x1"], S["d0b"], N, h2, w2, nm("h_a"))
        d_d0a = bw(L[3], d_d0b, S["d0b"], S["d0a"], N, h2, w2, nm("h_b"))
        d_x0 = bw(L[2], d_d0a, S["d0a"], S["x0"], N, H, W, nm("f_a"), residual=d_s0)
        d_a0 = bw(L[1], d_x0, S["x0"], S["a0"], N, H, W, nm("f_w"))
        return bw(L[0], d_a0, S["a0"], S["a_in"], N, H, W, nm("f_in"), want_dx=want_dx)

    # Row strips (forward_tiled).  Receptive field of one output row, measured on the float64 oracle (tests/test_ddnet_halo.py):
    # path 1 (temp1) -40..+37 rows, path 2 (pack, temp11 at half resolution, bilinear x2, fusion) -84..+78, temp2 -40..+37.
    STAGE_A_HALO = 88    # rows of the mosaic for both paths up to the temp2 input; a multiple of 8 (path 2 goes down by 8)
    STAGE_B_HALO = 40    # rows of the temp2 input (the U-shaped body, FastDVDnetEngine.BLOCK_HALO)
    # frame chunks: images x pixels of one path-1 body pass (3 images per centre frame).  The activations of a pass grow with
    # it (fp32 NHWC, 32..128 padded channels per level, three bodies); the budget keeps every size the tests and the
    # single-GPU benchmarks run in one pass and a 2048-wide strip of a 24-frame sequence in a few passes
    PASS_PIXELS = 1 << 24

    @classmethod
    def chunk_frames(cls, B, H, W):
        """Centre frames per pass for a B-frame sequence of H x W mosaics: at most PASS_PIXELS / (3 H W), the chunks made as
        even as that allows.  Every image's convolutions are the same whatever the chunk, so chunking changes no bit."""
        most = max(1, cls.PASS_PIXELS // (3 * H * W))
        n = -(-B // most)
        return -(-B // n)

    @classmethod
    def tiled_chunk_frames(cls, B, tile):
        """Chunk of forward_tiled: from the frame's global sizes (the longest halo-extended strip), so that every rank runs
        the same number of halo exchanges (P2PRegion counts them in lock-step)."""
        return cls.chunk_frames(B, min(tile.rows + 2 * cls.STAGE_A_HALO, tile.H_total), tile.W)

    @classmethod
    def check_tile(cls, tile):
        """Refuse strips forward_tiled cannot reproduce the whole frame on (before any GPU work)."""
        if tile.rows % 8 or tile.W % 8:
            raise ValueError("DDnet on row strips needs strips and width that are multiples of 8 (the half-resolution path "
                             "goes down by 8; strip starts must keep its stride phases), got %d rows x %d" % (tile.rows, tile.W))
        if tile.world > 1 and tile.rows < cls.STAGE_A_HALO:
            raise ValueError("DDnet on row strips: strips of %d rows are shorter than its %d-row halo (use fewer ranks for a "
                             "%d-row frame)" % (tile.rows, cls.STAGE_A_HALO, tile.H_total))

    def forward(self, mosaic, train=False):
        """mosaic [B,H,W] planar (whole circular sequence) -> demosaicked [B,3,H,W].  train=True keeps the activations.
        Inference runs the centre frames in chunks of ``chunk_frames`` (training in one pass: backward() needs it all)."""
        B, H, W = mosaic.shape
        if H % 8 or W % 8:
            raise NotImplementedError("native DDnet engine needs H, W multiples of 8 (half-resolution path with two "
                                      "stride-2 levels; the reference reflect-pads to 4, DDnet_test.py:180-187, and "
                                      "would itself fail on sizes that are not multiples of 8)")
        self.prepare(training=train)
        out = self.ws.get("dd_tr_out" if train else "dd_out", (B, 3, H, W), mosaic.device)
        Bc = B if train else self.chunk_frames(B, H, W)
        self.pdl_chain = (not train) and self.profile is None and self.impl == IMPL_TC      # see FastDVDnetEngine.forward
        try:
            for f0 in range(0, B, Bc):
                bc = min(Bc, B - f0)
                t2in, res1, res2 = self._stage_a(mosaic, f0, bc, Bc, 0, H, train)
                self._stage_b(t2in, res1, res2, bc, Bc, H, W, out[f0:f0 + bc], train)
        finally:
            self.pdl_chain = False
        if train:
            self._saved.update(mosaic=mosaic, B=B, H=H, W=W)
        return out

    def forward_tiled(self, mosaic_own, tile):
        """Inference on a row strip of a larger frame (``parallel.TileContext``): mosaic_own [B,rows,W], this rank's rows of
        the whole sequence -> demosaicked own rows [B,3,rows,W] (engine-owned buffer, valid until the next call).

        The mosaic is exchanged once with STAGE_A_HALO rows; per frame chunk both paths run on that extended strip up to the
        temp2 input, whose own rows are exchanged with STAGE_B_HALO rows (the packed NHWC rows as they are, viewed as
        [2Bc,1,rows,32W]); temp2 runs on that and the output mix on the own rows (res1 / res2 are used pixel-wise, they need
        no halo).  Extended strips start on global rows that are multiples of 8, so every stride phase is that of the whole
        frame, zero padding applies only at true image borders and the own rows are those of ``forward``."""
        B, rows, W = mosaic_own.shape
        self.prepare(training=False)
        m_ext, top = tile.exchange(mosaic_own.view(B, 1, rows, W), self.STAGE_A_HALO)
        m_ext = m_ext.view(B, m_ext.shape[2], W)
        out = self.ws.get("ddt_out", (B, 3, rows, W), mosaic_own.device)
        Bc = self.tiled_chunk_frames(B, tile)
        self.pdl_chain = self.profile is None and self.impl == IMPL_TC
        try:
            for f0 in range(0, B, Bc):
                bc = min(Bc, B - f0)
                t2in, res1, res2 = self._stage_a(m_ext, f0, bc, Bc, tile.r0 - top, tile.H_total, False)
                own = t2in[:, top:top + rows].contiguous().view(2 * bc, 1, rows, W * 32)
                t2_ext, top2 = tile.exchange(own, self.STAGE_B_HALO)
                self._stage_b(t2_ext.view(2 * bc, -1, W, 32), res1[:, :, top:top + rows].contiguous(),
                              res2[:, :, top:top + rows].contiguous(), bc, Bc, rows, W, out[f0:f0 + bc], False, top2)
        finally:
            self.pdl_chain = False
        return out

    def _stage_a(self, mosaic, f0, bc, cap, row0, H_total, train):
        """Both paths up to the temp2 input for the centre frames [f0, f0+bc) of mosaic [B,H,W], whose row 0 is row ``row0``
        of an ``H_total``-row frame.  Returns t2in [2bc,H,W,32] (path 1, then path 2), res1, res2 [bc,3,H,W]; buffers hold
        ``cap`` frames."""
        B, H, W = mosaic.shape
        dev = mosaic.device
        m = self.module
        a, a2 = m.weight_tensor_in.data, m.weight_tensor_in2.data
        sp = int(self.tf32)
        t = "tr_" if train else ""
        g = lambda name, k, shape: self.ws.get("dd_%s%s" % (t, name), (k * cap,) + shape, dev)[:k * bc]
        keep = (lambda tag: tag) if train else (lambda tag: None)
        t2in = g("t2in", 2, (H, W, 32))
        res1, res2 = g("res1", 1, (3, H, W)), g("res2", 1, (3, H, W))
        # path 1: full-resolution single-channel triples
        in1 = g("in1", 3, (H, W, 32))
        call("sci_ddnet_pack_input1_frames", ptr(mosaic), ptr(a), ptr(in1), B, f0, bc, H, W, 32, sp, stream())
        r1 = self._body(self.t1, in1, 3 * bc, H, W, keep=keep("t1"), cap=3 * cap)
        xo1, S1 = r1 if train else (r1, None)
        call("sci_ddnet_stage2_input_frames", ptr(mosaic), ptr(a), ptr(xo1), xo1.shape[-1], ptr(t2in), ptr(res1), B, f0, bc,
             H, W, 32, sp, stream())
        # path 2: half-resolution RGGB planes, residual, bilinear x2, fusion convs
        in4 = g("in4", 3, (H // 2, W // 2, 32))
        call("sci_ddnet_pack_input4_frames", ptr(mosaic), ptr(a2), ptr(in4), B, f0, bc, H, W, 32, sp, stream())
        r4 = self._body(self.t11, in4, 3 * bc, H // 2, W // 2, keep=keep("t11"), cap=3 * cap)
        xo4, S4 = r4 if train else (r4, None)
        up = g("up", 3, (H, W, 32))
        call("sci_ddnet_upsample4_strip", ptr(mosaic), ptr(a2), ptr(xo4), xo4.shape[-1], ptr(up), B, f0, bc, H, W, row0,
             H_total, 32, sp, stream())
        f0_ = g("f0", 3, (H, W, self.fus[0].out_ch))
        self.conv(self.fus[0], up, 3 * bc, H, W, f0_)
        xf = g("xf", 3, (H, W, self.fus[1].out_ch))
        self.conv(self.fus[1], f0_, 3 * bc, H, W, xf, round_out=False)
        call("sci_ddnet_stage2_input_frames", None, None, ptr(xf), xf.shape[-1], ptr(t2in[bc:]), ptr(res2), bc, 0, bc, H, W,
             32, sp, stream())
        self.n_launch += 5
        if train:
            self._saved = dict(S1=S1, S4=S4, up=up, f0=f0_, xf=xf, res1=res1, res2=res2)
        return t2in, res1, res2

    def _stage_b(self, t2in, res1, res2, bc, cap, rows, W, out, train, top=0):
        """temp2 on both paths (one batch of 2bc) and the learnable output mix of the ``rows`` rows from ``top`` on.
        t2in [2bc,top+rows+bot,W,32], res1 / res2 [bc,3,rows,W] -> out [bc,3,rows,W]."""
        Ht = t2in.shape[1]
        r2 = self._body(self.t2, t2in, 2 * bc, Ht, W, keep="t2" if train else None, cap=2 * cap)
        xo2, S2 = r2 if train else (r2, None)
        if Ht != rows:
            xo2 = xo2[:, top:top + rows].contiguous()
        a3 = self.module.weight_tensor_out.data
        call("sci_ddnet_output", ptr(res1), ptr(res2), ptr(xo2), xo2.shape[-1], ptr(a3), ptr(out), bc, rows, W, stream())
        self.n_launch += 1
        if train:
            self._saved.update(S2=S2, xo2=xo2)

    def backward(self, dout):
        """Gradients of ALL trained parameters (convs of temp1 / temp11 / fusion / temp2 and the three mixing tensors) into
        the flat grad bucket, given d loss / d output [B,3,H,W]."""
        sv = self._saved
        mosaic, B, H, W = sv["mosaic"], sv["B"], sv["H"], sv["W"]
        dev = dout.device
        m = self.module
        g = self.ws.get
        gv = self.bucket.grad_view
        da, da2, da3 = gv(m.weight_tensor_in), gv(m.weight_tensor_in2), gv(m.weight_tensor_out)
        da.zero_(); da2.zero_(); da3.zero_()
        self.begin_backward()
        # output mix and the two residual adds of temp2
        d_xo2 = g("ddg_xo2", (2 * B, H, W, 32), dev)
        d_res1, d_res2 = g("ddg_res1", (B, 3, H, W), dev), g("ddg_res2", (B, 3, H, W), dev)
        call("sci_ddnet_output_bwd", ptr(dout), ptr(sv["res1"]), ptr(sv["res2"]), ptr(sv["xo2"]), sv["xo2"].shape[-1],
             ptr(m.weight_tensor_out.data), ptr(d_xo2), ptr(d_res1), ptr(d_res2), ptr(da3), B, H, W, stream())
        d_t2in = self._body_backward(self.t2, sv["S2"], d_xo2, 2 * B, H, W, True, "t2")
        # path 1
        d_xo1 = g("ddg_xo1", (3 * B, H, W, 32), dev)
        call("sci_ddnet_stage2_input_bwd", ptr(d_t2in), ptr(d_res1), ptr(mosaic), ptr(d_xo1), ptr(da), B, H, W, stream())
        d_in1 = self._body_backward(self.t1, sv["S1"], d_xo1, 3 * B, H, W, True, "t1")
        call("sci_ddnet_pack_input1_bwd", ptr(d_in1), ptr(mosaic), ptr(da), B, H, W, stream())
        # path 2: fusion convs, bilinear up-sampling, residual, temp11
        d_xf = g("ddg_xf", (3 * B, H, W, 32), dev)
        call("sci_ddnet_stage2_input_bwd", ptr(d_t2in[B:]), ptr(d_res2), None, ptr(d_xf), None, B, H, W, stream())
        d_f0 = self._layer_bwd(self.fus[1], d_xf, None, sv["f0"], 3 * B, H, W, "ddg_f0")
        d_up = self._layer_bwd(self.fus[0], d_f0, sv["f0"], sv["up"], 3 * B, H, W, "ddg_up")
        d_y4 = g("ddg_y4", (3 * B, H // 2, W // 2, 32), dev, zero=True)
        call("sci_ddnet_upsample4_bwd", ptr(d_up), ptr(d_y4), B, H, W, stream())
        call("sci_ddnet_pack_input4_bwd", ptr(d_y4), ptr(mosaic), ptr(da2), B, H, W, 1, stream())
        d_in4 = self._body_backward(self.t11, sv["S4"], d_y4, 3 * B, H // 2, W // 2, True, "t11")
        call("sci_ddnet_pack_input4_bwd", ptr(d_in4), ptr(mosaic), ptr(da2), B, H, W, 0, stream())
        self.finish_param_grads()
        self.n_launch += 8

    def forward_window(self, x):
        """Reference call convention model(x[1,15,H,W]) for ONE 5-frame window (network_demosaicking.py:406-463);
        API parity only — the solvers use forward().  With B = 5 the centre frame 2 reads the frames 0..4 in order."""
        if x.shape[0] != 1 or x.shape[1] != 15:
            raise _lib.SciError("expected x of shape [1,15,H,W]")
        H, W = x.shape[2], x.shape[3]
        rgb = x.view(5, 3, H, W).contiguous().float()
        mosaic = self.ws.get("dd_win_mosaic", (5, H, W), rgb.device)
        call("sci_rgb_sum", ptr(rgb), ptr(mosaic), H, W, 5, stream())
        return self.forward(mosaic)[2:3].clone()
