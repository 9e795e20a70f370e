"""Network boundary kernels, one C-ABI entry point at a time.

The kernels between the tensor-core convolutions and the ADMM loop - the FFDNet / FastDVDnet / DDnet input packers and
output unpackers, DDnet's learnable scalars, residual adds, bilinear x2 and output mix, the losses, the adjoints of all
of these, and the stage-2 bookkeeping of sci_ops.cu - are called directly through ``_lib.call``.  sci_train.cu,
sci_ddnet.cu and sci_ops.cu are compiled with --fmad=false and without fast math, so every kernel here is a fixed
sequence of IEEE single-precision operations.  Four kinds of check:

A. Bit-exact against a float32 restatement in the kernel's op order: separate torch float32 ops on the CPU, TF32 splits
   as cvt.rna (ties away from zero), fp16 as round-to-nearest-even.  Inputs carry constructed TF32 ties (low 14 bits
   0x1000), and every split case whose ties reach the rounding asserts that a ties-to-even restatement differs.
B. Semantics against an independent float64 statement (F.pixel_unshuffle / pixel_shuffle, torch.roll for the circular
   frame windows, F.interpolate(bilinear, align_corners=True), the mean-square formulas): per element
   |got - ref| <= n 2^-24 S, n the fp32 roundings on the element's path and S the float64 sum of |terms|.  Remaps are
   the case n = 0.  A TF32 value + remainder pair adds 2^-22 |v|, an fp16 one 2^-22 |v| plus its subnormal spacing.
C. Reductions with atomics (da, da2, da3, act_bwd's s1 / s2, the losses, sse, the scatter of upsample4_bwd) against
   float64 within (depth) 2^-24 S, depth the chain actually used: the roundings that form a term, the 8 levels of the
   256-thread shuffle tree (or act_bwd's grid-stride passes and row loop), and one atomic add per block in any order.
D. Adjoints equal torch.autograd.grad of the float64 forward of B with respect to the same inputs: bit-exact where the
   adjoint is a copy, a negation or one fp32 product or sum of two (float64, rounded once), within C's bound where it
   sums.  Accumulating outputs are prefilled with nonzero values and must be added to.

Every bound has teeth: a perturbed float64 reference (a wrong channel order, window offset or scalar index, the other
align_corners convention, or the last ragged block of pixels / one frame's contributions left out) must violate it.
Operands of the reductions are positive (in [0.5, 1]), so no term can cancel and a missing block moves the sum far
past the bound.  Outputs are prefilled with NaN inside sentinel margins: every written element must be finite, every
margin untouched, padded channels exactly 0.  Input columns no kernel may read hold NaN.  Every bounded check prints
max and RMS of err / bound (pytest -s).  The CPU-only cases run each float32 restatement against its float64 statement,
with the same bounds and teeth, without a device."""
import math
import zlib

import pytest
import torch
import torch.nn.functional as F

from test_gpu_conv_plans import _bits, _guarded, _margins_intact, _report, tf32

gpu = pytest.mark.gpu
U = 2.0 ** -24
TREE = 8                    # levels of the 256-thread shuffle tree of every block reduction
H_, W_ = 38, 70             # 2660 pixels = 10 blocks of 256 + 100; half resolution 19 x 35 = 665 pixels (35: no multiple of 32)
SIGMA = 25.0 / 255.0
NAN = float("nan")


# ---- inputs and rounding ---------------------------------------------------------------------------------------------
def _gen(*key):
    return torch.Generator().manual_seed(zlib.crc32(repr(key).encode()))


def _pos(g, *shape):
    return 0.5 + 0.5 * torch.rand(shape, generator=g)


def _ties(t, g, frac=0.25):
    """Constructed TF32 ties: low 14 bits 0x1000 (bit 13 clear), where ties-away and ties-to-even round apart."""
    i = t.clone().view(torch.int32)
    sel = torch.rand(t.shape, generator=g) < frac
    i[sel] = (i[sel] & -16384) | 0x1000
    return i.view(torch.float32)


def tf32_rne(t):
    """TF32 rounding with ties to even: the wrong mode, which the tie inputs must tell apart from cvt.rna."""
    i = t.contiguous().view(torch.int32)
    return ((i + 0xFFF + ((i >> 13) & 1)) & -8192).view(torch.float32)


def _put(dst, k, v, split, tf=tf32):
    """Channels k.. <- v; split: TF32 value in k.., TF32 remainder in k+16.. (put() of sci_ddnet.cu, the packers)."""
    n = v.shape[-1]
    if split:
        hi = tf(v)
        dst[..., k:k + n] = hi
        dst[..., 16 + k:16 + k + n] = tf(v - hi)
    else:
        dst[..., k:k + n] = v


def _nan_cols(t, k):
    t = t.clone()
    t[..., k:] = NAN
    return t


def _blocks(n, b=256):
    return (n + b - 1) // b


# ---- checks --------------------------------------------------------------------------------------------------------
def _run(name, *args):
    from adaptivepnp_sci_b200 import _lib as L
    L.call(name, *[L.ptr(a) if a is None or isinstance(a, torch.Tensor) else a for a in args], L.stream())
    torch.cuda.synchronize()


def _dev_out(shape, dev, init=None, dtype=torch.float32):
    buf, t = _guarded(shape, dtype, dev)
    if init is not None:
        t.copy_(init)
    return buf, t


def _intact(tag, *bufs):
    for b in bufs:
        assert _margins_intact(b), "%s: wrote outside its output" % tag


def _exact(tag, got, want):
    got = got.detach().cpu()
    want = want.detach().cpu().to(got.dtype)
    assert bool(torch.isfinite(got.float()).all()), "%s: non-finite output" % tag
    diff = _bits(got) != _bits(want)
    assert not bool(diff.any()), "%s: %d of %d elements differ bit-wise" % (tag, int(diff.sum()), diff.numel())


def _bounded(tag, got, ref, eb, teeth=()):
    """|got - ref| <= eb per element; every (what, perturbed reference) in teeth must violate the bound somewhere."""
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    eb = (eb.detach() if isinstance(eb, torch.Tensor) else torch.tensor(eb)).double().cpu().expand_as(ref)
    assert bool(torch.isfinite(got).all()), "%s: non-finite output" % tag
    err = (got - ref).abs()
    pos = eb > 0
    if bool(pos.any()):
        _report(tag, err[pos], eb[pos])
    bad = err > eb
    assert not bool(bad.any()), "%s: %d of %d elements beyond the bound, max err %.3g" % (
        tag, int(bad.sum()), bad.numel(), float(err.max()))
    for what, t in teeth:
        assert bool(((t.detach().double().cpu() - ref).abs() > eb).any()), "%s: the bound cannot see %s" % (tag, what)


def _sum_bound(S, depth):
    return depth * U * S


# ---- FFDNet: pixel-(un)shuffle + sigma map --------------------------------------------------------------------------
def _unshuffle32(u):
    """[B][C][H][W] -> [B][H/2][W/2][4C], channel c*4 + dy*2 + dx."""
    B, C, H, W = u.shape
    return u.reshape(B, C, H // 2, 2, W // 2, 2).permute(0, 2, 4, 1, 3, 5).reshape(B, H // 2, W // 2, 4 * C)


def _shuffle32(y, C):
    B, h2, w2, _ = y.shape
    return y[..., :4 * C].reshape(B, h2, w2, C, 2, 2).permute(0, 3, 1, 4, 2, 5).reshape(B, C, 2 * h2, 2 * w2)


def _swap_dydx(t, C):
    return t.reshape(*t.shape[:-1], C, 2, 2).transpose(-1, -2).reshape(t.shape)


def r_ffdnet_pack(u, sigma, Cpad, rnd, tf=tf32):
    B, C, H, W = u.shape
    v = torch.zeros(B, H // 2, W // 2, Cpad)
    v[..., :4 * C] = _unshuffle32(u)
    v[..., 4 * C] = sigma
    if rnd:
        lo = v[..., :16].clone()
        v[..., 16:] = 0
        _put(v, 0, lo, 1, tf)
    return v


def case_ffdnet_pack(dev, C, rnd, Cpad, B=2, H=H_, W=W_):
    g = _gen("ffdnet_pack", C, rnd, Cpad, B, H, W)
    u = _ties(_pos(g, B, C, H, W), g)
    want = r_ffdnet_pack(u, SIGMA, Cpad, rnd)
    got = want
    if dev is not None:
        buf, out = _dev_out((B, H // 2, W // 2, Cpad), dev)
        _run("sci_ffdnet_pack_input", u.to(dev), SIGMA, out, B, C, H, W, Cpad, rnd)
        _intact("ffdnet_pack_input", buf)
        got = out.cpu()
        _exact("ffdnet_pack_input", got, want)
    if rnd:
        assert not torch.equal(_bits(got), _bits(r_ffdnet_pack(u, SIGMA, Cpad, rnd, tf32_rne))), "ties to even not told apart"
    used = set(range(4 * C + 1)) | ({16 + k for k in range(4 * C + 1)} if rnd else set())
    assert bool((got[..., [k for k in range(Cpad) if k not in used]] == 0).all()), "padded channels must be 0"
    ref = torch.cat([F.pixel_unshuffle(u.double(), 2).permute(0, 2, 3, 1),
                     torch.full((B, H // 2, W // 2, 1), float(torch.tensor(SIGMA)), dtype=torch.float64)], -1)
    val = got[..., :4 * C + 1].double() + (got[..., 16:17 + 4 * C].double() if rnd else 0)
    bad = ref.clone()
    bad[..., :4 * C] = _swap_dydx(ref[..., :4 * C], C)
    _bounded("ffdnet_pack_input C=%d rnd=%d Cpad=%d" % (C, rnd, Cpad), val, ref, 4 * U * ref.abs() if rnd else 0.0,
             [("dy / dx swapped", bad)])


def case_ffdnet_unpack(dev, C, Cpad, B=2, H=H_, W=W_):
    """unpack and its adjoint on 8-bit dyadic values, so that <unpack(y), g> = <y, unpack_grad(g)> holds exactly."""
    g = _gen("ffdnet_unpack", C, Cpad, B, H, W)
    y = torch.round((2 * torch.rand(B, H // 2, W // 2, Cpad, generator=g) - 1) * 256) / 256
    y = _nan_cols(y, 4 * C)
    dx = torch.round((2 * torch.rand(B, C, H, W, generator=g) - 1) * 256) / 256
    want_x = _shuffle32(y, C)
    want_dy = torch.zeros(B, H // 2, W // 2, Cpad)
    want_dy[..., :4 * C] = _unshuffle32(dx)
    got_x, got_dy = want_x, want_dy
    if dev is not None:
        bx, ox = _dev_out((B, C, H, W), dev)
        bd, od = _dev_out((B, H // 2, W // 2, Cpad), dev)
        _run("sci_ffdnet_unpack_output", y.to(dev), ox, B, C, H, W, Cpad)
        _run("sci_ffdnet_unpack_output_grad", dx.to(dev), od, B, C, H, W, Cpad)
        _intact("ffdnet_unpack", bx, bd)
        got_x, got_dy = ox.cpu(), od.cpu()
        _exact("ffdnet_unpack_output", got_x, want_x)
        _exact("ffdnet_unpack_output_grad", got_dy, want_dy)
    y64 = y.double().nan_to_num(0.0).requires_grad_()
    ref_x = F.pixel_shuffle(y64[..., :4 * C].permute(0, 3, 1, 2), 2)
    bad = F.pixel_shuffle(_swap_dydx(y64[..., :4 * C], C).permute(0, 3, 1, 2), 2)
    _bounded("ffdnet_unpack_output", got_x, ref_x, 0.0, [("dy / dx swapped", bad)])
    (ref_dy,) = torch.autograd.grad(ref_x, y64, dx.double())
    _bounded("ffdnet_unpack_output_grad", got_dy, ref_dy, 0.0)
    assert bool((got_dy[..., 4 * C:] == 0).all()), "padded channels must be 0"
    lhs = float((got_x.double() * dx.double()).sum())
    rhs = float((y[..., :4 * C].double() * got_dy[..., :4 * C].double()).sum())
    assert lhs == rhs, "adjoint identity: %r != %r" % (lhs, rhs)


def r_split_pack(u, sigma):
    B, C, H, W = u.shape
    v = torch.zeros(B, H // 2, W // 2, 32)
    v[..., :4 * C] = _unshuffle32(u)
    v[..., 4 * C] = sigma
    hi = v.half()
    return torch.cat([hi, ((v - hi.float()) * 2048.0).half()], -1)


def r_split_unpack(y, C):
    # fmaf(rem, 2^-11, hi): the product is exact, so one rounding, as in the separate ops here
    return _shuffle32(y[..., 32:].float() * (1.0 / 2048.0) + y[..., :32].float(), C)


def case_ffdnet_split_half(dev, C, B=2, H=H_, W=W_):
    g = _gen("ffdnet_split", C, B, H, W)
    u = torch.rand(B, C, H, W, generator=g)
    r = torch.rand(B, C, H, W, generator=g)
    u = torch.where(r < 0.3, u * 6e-5, torch.where(r < 0.6, 700.0 + 300.0 * u, u))      # fp16 subnormals, values near 10^3
    want_p = r_split_pack(u, SIGMA)
    got_p = want_p
    if dev is not None:
        bp, op = _dev_out((B, H // 2, W // 2, 64), dev, dtype=torch.float16)
        _run("sci_ffdnet_pack_input_split_half", u.to(dev), SIGMA, op, B, C, H, W)
        bx, ox = _dev_out((B, C, H, W), dev)
        _run("sci_ffdnet_unpack_output_split_half", op, ox, B, C, H, W)
        _intact("ffdnet_split_half", bp, bx)
        got_p, got_x = op.cpu(), ox.cpu()
        _exact("ffdnet_pack_input_split_half", got_p, want_p)
        _exact("ffdnet_unpack_output_split_half", got_x, r_split_unpack(got_p, C))
    else:
        got_x = r_split_unpack(got_p, C)
    hi = got_p[..., :32]
    assert bool(((hi != 0) & (hi.float().abs() < 2.0 ** -14)).any()), "no fp16 subnormal reached"
    assert bool((got_p[..., 4 * C + 1:32] == 0).all()) and bool((got_p[..., 33 + 4 * C:] == 0).all()), "padded channels"
    ref = _unshuffle32(u.double())
    eb = (2.0 ** -22) * ref.abs() + 2.0 ** -36
    val = got_p[..., :4 * C].double() + got_p[..., 32:32 + 4 * C].double() / 2048
    _bounded("ffdnet_pack_input_split_half C=%d" % C, val, ref, eb, [("the remainder left out", got_p[..., :4 * C])])
    y64 = got_p[..., :32].double() + got_p[..., 32:].double() / 2048
    ref_x = F.pixel_shuffle(y64[..., :4 * C].permute(0, 3, 1, 2), 2)
    _bounded("ffdnet_unpack_output_split_half C=%d" % C, got_x, ref_x, U * ref_x.abs(),
             [("the remainder left out", F.pixel_shuffle(got_p[..., :4 * C].double().permute(0, 3, 1, 2), 2))])
    # round trip: 2^-22 |u| from the split, 2^-36 from a subnormal remainder, 2^-24 |u| from the final rounding
    _bounded("ffdnet split round trip C=%d" % C, got_x, u.double(), (2.0 ** -22 + U) * u.double().abs() + 2.0 ** -36,
             [("the remainder left out", _shuffle32(got_p[..., :32].double(), C))])


# ---- FastDVDnet: circular frame triples + residual output ------------------------------------------------------------
def _slot_src(B, s):
    return [(f + s - 1) % B for f in range(B)]


def r_fdvd_pack(frames, sigma, Cpad, rnd, tf=tf32):
    B, _, H, W = frames.shape
    P = H * W
    out = torch.zeros(B, P, Cpad)
    for s in range(3):
        blk = torch.cat([frames[_slot_src(B, s)].reshape(B, 3, P).permute(0, 2, 1), torch.full((B, P, 1), sigma)], -1)
        _put(out, 4 * s, blk, rnd, tf)
    return out


def _fdvd_ref64(frames64, sigma, Cpad, shift=1):
    """float64 input block, [B][P][Cpad]: slot s of centre frame f = frame (f + s - 1) mod B (torch.roll), then sigma."""
    B, _, H, W = frames64.shape
    P = H * W
    cols = []
    for s in range(3):
        cols += [torch.roll(frames64, shift - s, 0).reshape(B, 3, P).permute(0, 2, 1),
                 torch.full((B, P, 1), float(torch.tensor(sigma)), dtype=torch.float64)]
    cols.append(torch.zeros(B, P, Cpad - 12, dtype=torch.float64))
    return torch.cat(cols, -1)


def case_fdvd_pack(dev, Cpad, rnd, B, H=H_, W=W_):
    g = _gen("fdvd_pack", Cpad, rnd, B, H, W)
    frames = _ties(_pos(g, B, 3, H, W), g)
    want = r_fdvd_pack(frames, SIGMA, Cpad, rnd)
    got = want
    if dev is not None:
        buf, out = _dev_out((B, H * W, Cpad), dev)
        _run("sci_fastdvd_pack_input", frames.to(dev), SIGMA, out, B, H, W, Cpad, rnd)
        _intact("fastdvd_pack_input", buf)
        got = out.cpu()
        _exact("fastdvd_pack_input", got, want)
    if rnd:
        assert not torch.equal(_bits(got), _bits(r_fdvd_pack(frames, SIGMA, Cpad, rnd, tf32_rne))), "ties to even not told apart"
    used = set(range(12)) | (set(range(16, 28)) if rnd else set())
    assert bool((got[..., [k for k in range(Cpad) if k not in used]] == 0).all()), "padded channels must be 0"
    ref = _fdvd_ref64(frames.double(), SIGMA, Cpad)[..., :12]
    val = got[..., :12].double() + (got[..., 16:28].double() if rnd else 0)
    teeth = [("colour channels reversed",
              torch.cat([torch.cat([ref[..., 4 * s:4 * s + 3].flip(-1), ref[..., 4 * s + 3:4 * s + 4]], -1) for s in range(3)], -1))]
    if B > 1:
        teeth.append(("the window shifted by one frame", _fdvd_ref64(frames.double(), SIGMA, Cpad, shift=2)[..., :12]))
    _bounded("fastdvd_pack_input Cpad=%d rnd=%d B=%d" % (Cpad, rnd, B), val, ref, 4 * U * ref.abs() if rnd else 0.0, teeth)


def r_fdvd_half(frames, sigma, C, scale=1.0):
    B, _, H, W = frames.shape
    P = H * W
    out = torch.zeros(B, P, C, dtype=torch.float16)
    for s in range(3):
        blk = torch.cat([frames[_slot_src(B, s)].reshape(B, 3, P).permute(0, 2, 1), torch.full((B, P, 1), sigma)], -1)
        hi = blk.half()
        out[..., 4 * s:4 * s + 4] = hi
        out[..., 16 + 4 * s:20 + 4 * s] = ((blk - hi.float()) * scale).half()
    return out


def case_fdvd_half(dev, C, B, H=H_, W=W_):
    g = _gen("fdvd_half", C, B, H, W)
    frames = _pos(g, B, 3, H, W)
    want = r_fdvd_half(frames, SIGMA, C)
    got = want
    if dev is not None:
        buf, out = _dev_out((B, H * W, C), dev, dtype=torch.float16)
        _run("sci_fastdvd_pack_input_half", frames.to(dev), SIGMA, out, B, H, W, C)
        _intact("fastdvd_pack_input_half", buf)
        got = out.cpu()
        _exact("fastdvd_pack_input_half", got, want)
    assert not torch.equal(_bits(got), _bits(r_fdvd_half(frames, SIGMA, C, 2048.0))), "remainder must not carry the 2^11 scale"
    pad = [k for k in range(C) if not (k < 12 or 16 <= k < 28)]
    assert bool((got[..., pad] == 0).all()), "padded channels must be 0"
    ref = _fdvd_ref64(frames.double(), SIGMA, 12)
    val = got[..., :12].double() + got[..., 16:28].double()
    # fp16 remainder without a scale: 2^-22 |v| where it is normal, its subnormal spacing 2^-24 / 2 where it is not
    _bounded("fastdvd_pack_input_half C=%d B=%d" % (C, B), val, ref, 2.0 ** -22 * ref.abs() + 2.0 ** -25,
             [("the remainder left out", got[..., :12])])


def r_fdvd_pack_grad(din, init, B):
    v = init.clone()
    for s in range(3):
        v = v + din[[(j - s + 1) % B for j in range(B)]][..., 4 * s:4 * s + 3].permute(0, 2, 1)
    return v


def case_fdvd_pack_grad(dev, B, acc, Cpad=16, H=H_, W=W_):
    g = _gen("fdvd_pack_grad", B, acc, Cpad, H, W)
    P = H * W
    din = _pos(g, B, P, Cpad)
    din[..., [3, 7, 11]] = NAN                       # sigma columns: no gradient flows to the frames
    din = _nan_cols(din, 12)
    init = _pos(g, B, 3, P) if acc else torch.zeros(B, 3, P)
    want = r_fdvd_pack_grad(din, init, B)
    got = want
    if dev is not None:
        buf, out = _dev_out((B, 3, P), dev, init if acc else None)
        _run("sci_fastdvd_pack_input_grad", din.to(dev), out, B, H, W, Cpad, acc)
        _intact("fastdvd_pack_input_grad", buf)
        got = out.cpu()
        _exact("fastdvd_pack_input_grad", got, want)
    fr64 = torch.zeros(B, 3, H, W, dtype=torch.float64, requires_grad=True)
    d64 = din.double().nan_to_num(0.0)

    def adj(d):
        return torch.autograd.grad(_fdvd_ref64(fr64, SIGMA, Cpad), fr64, d, retain_graph=True)[0].reshape(B, 3, P)
    ref = init.double() + adj(d64)
    S = init.double() + adj(d64.abs())
    d0 = d64.clone()
    d0[0] = 0
    _bounded("fastdvd_pack_input_grad B=%d acc=%d" % (B, acc), got, ref, _sum_bound(S, 3),
             [("centre frame 0's window left out", init.double() + adj(d0))])


def case_fdvd_output(dev, Cpad, B, H=H_, W=W_):
    g = _gen("fdvd_output", Cpad, B, H, W)
    P = H * W
    frames = _pos(g, B, 3, H, W)
    y = _nan_cols(_pos(g, B, P, Cpad), 3)
    dout = 2 * torch.rand(B, 3, H, W, generator=g) - 1
    want_o = (frames.reshape(B, 3, P) - y[..., :3].permute(0, 2, 1)).reshape(B, 3, H, W)
    want_d = torch.zeros(B, P, Cpad)
    want_d[..., :3] = -dout.reshape(B, 3, P).permute(0, 2, 1)
    got_o, got_d = want_o, want_d
    if dev is not None:
        bo, oo = _dev_out((B, 3, H, W), dev)
        bd, od = _dev_out((B, P, Cpad), dev)
        _run("sci_fastdvd_output", frames.to(dev), y.to(dev), oo, B, H, W, Cpad)
        _run("sci_fastdvd_output_grad", dout.to(dev), od, B, H, W, Cpad)
        _intact("fastdvd_output", bo, bd)
        got_o, got_d = oo.cpu(), od.cpu()
        _exact("fastdvd_output", got_o, want_o)
        _exact("fastdvd_output_grad", got_d, want_d)
    y64 = y.double().nan_to_num(0.0).requires_grad_()
    ref = frames.double() - y64[..., :3].permute(0, 2, 1).reshape(B, 3, H, W)
    bad = frames.double() - y64[..., :3].flip(-1).permute(0, 2, 1).reshape(B, 3, H, W)
    _bounded("fastdvd_output Cpad=%d" % Cpad, got_o, ref, U * (frames.double() + y64[..., :3].permute(0, 2, 1).reshape(B, 3, H, W)),
             [("colour channels reversed", bad)])
    (ref_d,) = torch.autograd.grad(ref, y64, dout.double())
    _bounded("fastdvd_output_grad Cpad=%d" % Cpad, got_d, ref_d, 0.0)
    assert bool((got_d[..., 3:] == 0).all()), "padded channels must be 0"


def case_fdvd_noisy(dev, n=3 * 2660 + 1):
    g = _gen("noisy", n)
    v = torch.rand(n, generator=g)
    noise = torch.randn(n, generator=g, dtype=torch.float64) * 0.1
    want = v + (v.double() + noise).float()
    got = want
    if dev is not None:
        buf, out = _dev_out((n,), dev)
        _run("sci_fastdvd_noisy_input", v.to(dev), noise.to(dev), out, n)
        _intact("fastdvd_noisy_input", buf)
        got = out.cpu()
        _exact("fastdvd_noisy_input", got, want)
    v64 = v.double()
    _bounded("fastdvd_noisy_input", got, 2 * v64 + noise, 2.01 * U * (2 * v64.abs() + noise.abs()),
             [("the measurement added once", v64 + noise)])


# ---- DDnet -----------------------------------------------------------------------------------------------------------
def _scalars(g, n):
    a = _pos(g, n)
    a[::4] = torch.tensor([0.5, 1.0, 2.0, 0.25, 4.0, 0.5, 1.0, 2.0, 0.5])[:len(a[::4])]    # powers of two keep the ties
    return a


def _src(B, off):
    return [(f + off) % B for f in range(B)]


def r_dd_pack1(m, a, split, tf=tf32):
    B = m.shape[0]
    mf = m.reshape(B, -1)
    out = torch.zeros(3 * B, mf.shape[1], 32)
    for j in range(3):
        for k in range(3):
            _put(out[j * B:(j + 1) * B], k, (mf[_src(B, j + k - 2)] * a[3 * j + k])[..., None], split, tf)
    return out


def _dd_pack1_64(m64, a64, swap=False, shift=2):
    B = m64.shape[0]
    cols = [[torch.roll(m64, shift - j - k, 0).reshape(B, -1, 1) * a64[3 * k + j if swap else 3 * j + k] for k in range(3)]
            for j in range(3)]
    return torch.cat([torch.cat(c, -1) for c in cols], 0)          # [3B][P][3]


def _quad(m):
    """[B][H][W] -> [B][H/2 * W/2][4], ib = dy*2 + dx."""
    B, H, W = m.shape
    return m.reshape(B, H // 2, 2, W // 2, 2).permute(0, 1, 3, 2, 4).reshape(B, -1, 4)


def _quad64(m64):
    B = m64.shape[0]
    return F.pixel_unshuffle(m64[:, None], 2).permute(0, 2, 3, 1).reshape(B, -1, 4)


def r_dd_pack4(m, a2, split, tf=tf32):
    B = m.shape[0]
    q = _quad(m)
    out = torch.zeros(3 * B, q.shape[1], 32)
    for j in range(3):
        for k in range(3):
            _put(out[j * B:(j + 1) * B], 4 * k, q[_src(B, j + k - 2)] * a2[(3 * j + k) * 4:(3 * j + k) * 4 + 4], split, tf)
    return out


def _dd_pack4_64(m64, a64, ks=(0, 1, 2), swap=False):
    B = m64.shape[0]
    rows = []
    for j in range(3):
        rows.append(torch.cat([_quad64(torch.roll(m64, 2 - j - k, 0)) *
                               a64[(3 * k + j if swap else 3 * j + k) * 4:(3 * k + j if swap else 3 * j + k) * 4 + 4]
                               for k in ks], -1))
    return torch.cat(rows, 0)                                       # [3B][hp][4 len(ks)]


def case_dd_pack(dev, B, split, H=H_, W=W_):
    g = _gen("dd_pack", B, split, H, W)
    m = _ties(_pos(g, B, H, W), g)
    a, a2 = _scalars(g, 9), _scalars(g, 36)
    want1, want4 = r_dd_pack1(m, a, split), r_dd_pack4(m, a2, split)
    got1, got4 = want1, want4
    if dev is not None:
        b1, o1 = _dev_out(want1.shape, dev)
        b4, o4 = _dev_out(want4.shape, dev)
        md = m.to(dev)
        _run("sci_ddnet_pack_input1", md, a.to(dev), o1, B, H, W, 32, split)
        _run("sci_ddnet_pack_input4", md, a2.to(dev), o4, B, H, W, 32, split)
        _intact("ddnet_pack_input", b1, b4)
        got1, got4 = o1.cpu(), o4.cpu()
        _exact("ddnet_pack_input1", got1, want1)
        _exact("ddnet_pack_input4", got4, want4)
    if split:
        assert not torch.equal(_bits(got1), _bits(r_dd_pack1(m, a, split, tf32_rne))), "ties to even not told apart"
        assert not torch.equal(_bits(got4), _bits(r_dd_pack4(m, a2, split, tf32_rne))), "ties to even not told apart"
    for got, n in ((got1, 3), (got4, 12)):
        used = set(range(n)) | (set(range(16, 16 + n)) if split else set())
        assert bool((got[..., [k for k in range(32) if k not in used]] == 0).all()), "padded channels must be 0"
    m64 = m.double()
    for tag, got, n, ref, bad in (
            ("ddnet_pack_input1", got1, 3, _dd_pack1_64(m64, a.double()), _dd_pack1_64(m64, a.double(), swap=True)),
            ("ddnet_pack_input4", got4, 12, _dd_pack4_64(m64, a2.double()), _dd_pack4_64(m64, a2.double(), swap=True))):
        val = got[..., :n].double() + (got[..., 16:16 + n].double() if split else 0)
        _bounded("%s B=%d split=%d" % (tag, B, split), val, ref, (1 + 4 * split) * U * ref.abs(),
                 [("the scalars of slot and triple exchanged", bad)])
    if B > 1:
        _bounded("ddnet_pack_input1 window", got1[..., :3].double() + (got1[..., 16:19].double() if split else 0),
                 _dd_pack1_64(m64, a.double()), (1 + 4 * split) * U * _dd_pack1_64(m64, a.double()).abs(),
                 [("the window shifted by one frame", _dd_pack1_64(m64, a.double(), shift=3))])


def r_dd_mid(m, a, xo, split, tf=tf32):
    B = xo.shape[0] // 3
    P = xo.shape[1]
    t2 = torch.zeros(B, P, 32)
    res = None
    for j in range(3):
        y = xo[j * B:(j + 1) * B, :, :3]
        v = y if m is None else (m.reshape(B, P)[_src(B, j - 1)] * a[3 * j + 1])[..., None] + y
        _put(t2, 3 * j, v, split, tf)
        if j == 1:
            res = v.permute(0, 2, 1).contiguous()
    return t2, res


def _dd_mid64(m64, a64, xo64, ai=1):
    """float64 temp2 input per triple, [3][B][P][3], and the |terms| sum S."""
    B = xo64.shape[0] // 3
    vs, ss = [], []
    for j in range(3):
        y = xo64[j * B:(j + 1) * B, :, :3]
        if m64 is None:
            vs.append(y)
            ss.append(y.abs())
        else:
            in1 = torch.roll(m64, 1 - j, 0).reshape(B, -1, 1) * a64[3 * j + ai]
            vs.append(in1 + y)
            ss.append(in1.abs() + y.abs())
    return torch.stack(vs), torch.stack(ss)


def case_dd_mid(dev, B, split, xo_cpad, path1, H=H_, W=W_):
    g = _gen("dd_mid", B, split, xo_cpad, path1, H, W)
    P = H * W
    m = _pos(g, B, H, W) if path1 else None
    a = _scalars(g, 9) if path1 else None
    xo = _nan_cols(_ties(_pos(g, 3 * B, P, xo_cpad), g), 3)
    want_t, want_r = r_dd_mid(m, a, xo, split)
    got_t, got_r = want_t, want_r
    if dev is not None:
        bt, ot = _dev_out((B, P, 32), dev)
        br, orr = _dev_out((B, 3, P), dev)
        _run("sci_ddnet_stage2_input", None if m is None else m.to(dev), None if a is None else a.to(dev), xo.to(dev), xo_cpad,
             ot, orr, B, H, W, 32, split)
        _intact("ddnet_stage2_input", bt, br)
        got_t, got_r = ot.cpu(), orr.cpu()
        _exact("ddnet_stage2_input t2in", got_t, want_t)
        _exact("ddnet_stage2_input res", got_r, want_r)
    if split and not path1:
        assert not torch.equal(_bits(got_t), _bits(r_dd_mid(m, a, xo, split, tf32_rne)[0])), "ties to even not told apart"
    used = set(range(9)) | (set(range(16, 25)) if split else set())
    assert bool((got_t[..., [k for k in range(32) if k not in used]] == 0).all()), "padded channels must be 0"
    m64 = None if m is None else m.double()
    a64 = None if a is None else a.double()
    v64, S = _dd_mid64(m64, a64, xo.double())
    ref = torch.cat(list(v64), -1)
    Sc = torch.cat(list(S), -1)
    val = got_t[..., :9].double() + (got_t[..., 16:25].double() if split else 0)
    n = 2 if path1 else 0
    if path1:
        bad = torch.cat(list(_dd_mid64(m64, a64, xo.double(), ai=0)[0]), -1)
    else:
        bad = torch.cat([v.flip(-1) for v in v64], -1)
    tag = "ddnet_stage2_input B=%d split=%d xo_cpad=%d path%d" % (B, split, xo_cpad, 1 if path1 else 2)
    _bounded(tag, val, ref, (n + 4 * split) * U * Sc, [("the wrong scalar" if path1 else "colour channels reversed", bad)])
    _bounded(tag + " res", got_r, v64[1].permute(0, 2, 1), n * U * S[1].permute(0, 2, 1),
             [("the wrong triple", v64[0].permute(0, 2, 1))])


def _up_coords(n, n2):
    """fp32 source index and weights of the align_corners bilinear x2, as dd_up4_kernel computes them."""
    s = torch.tensor(float(n2 - 1)) / torch.tensor(float(n - 1))
    r = s * torch.arange(n, dtype=torch.float32)
    i0 = torch.clamp(r.to(torch.int64), max=n2 - 1)
    i1 = torch.clamp(i0 + 1, max=n2 - 1)
    l1 = torch.clamp(r - i0.float(), 0.0, 1.0)
    return i0, i1, 1.0 - l1, l1


def r_dd_up4(m, a2, xo4, split, H, W, tf=tf32):
    B = m.shape[0]
    h2, w2 = H // 2, W // 2
    q = _quad(m)
    out = torch.zeros(3 * B, H * W, 32)
    y0, y1, ly0, ly1 = _up_coords(H, h2)
    x0, x1, lx0, lx1 = _up_coords(W, w2)
    LY0, LY1 = ly0.view(1, H, 1, 1), ly1.view(1, H, 1, 1)
    LX0, LX1 = lx0.view(1, 1, W, 1), lx1.view(1, 1, W, 1)
    for j in range(3):
        val = (q[_src(B, j - 1)] * a2[(3 * j + 1) * 4:(3 * j + 2) * 4] + xo4[j * B:(j + 1) * B, :, :4]).reshape(B, h2, w2, 4)

        def at(yy, xx):
            return val[:, yy][:, :, xx]
        r0 = LX0 * at(y0, x0) + LX1 * at(y0, x1)
        r1 = LX0 * at(y1, x0) + LX1 * at(y1, x1)
        _put(out[j * B:(j + 1) * B], 0, (LY0 * r0 + LY1 * r1).reshape(B, H * W, 4), split, tf)
    return out


def _y4_64(m64, a64, xo4_64, H, W, k=1):
    """float64 y4 = centre slot of the path-2 input + the body's output, [3B][4][H/2][W/2], and its |terms|."""
    B = m64.shape[0]
    h2, w2 = H // 2, W // 2
    ys, ss = [], []
    for j in range(3):
        in1 = F.pixel_unshuffle(torch.roll(m64, 1 - j, 0)[:, None], 2) * a64[(3 * j + k) * 4:(3 * j + k + 1) * 4].view(1, 4, 1, 1)
        xb = xo4_64[j * B:(j + 1) * B, :, :4].reshape(B, h2, w2, 4).permute(0, 3, 1, 2)
        ys.append(in1 + xb)
        ss.append(in1.abs() + xb.abs())
    return torch.cat(ys, 0), torch.cat(ss, 0)


def _up64(y4, H, W, align=True):
    n = y4.shape[0]
    return F.interpolate(y4, size=(H, W), mode="bilinear", align_corners=align).permute(0, 2, 3, 1).reshape(n, H * W, 4)


def case_dd_up4(dev, B, split, xo_cpad, H=H_, W=W_):
    g = _gen("dd_up4", B, split, xo_cpad, H, W)
    h2, w2 = H // 2, W // 2
    m = _pos(g, B, H, W)
    a2 = _scalars(g, 36)
    xo4 = _nan_cols(_pos(g, 3 * B, h2 * w2, xo_cpad), 4)
    want = r_dd_up4(m, a2, xo4, split, H, W)
    got = want
    if dev is not None:
        buf, out = _dev_out((3 * B, H * W, 32), dev)
        _run("sci_ddnet_upsample4", m.to(dev), a2.to(dev), xo4.to(dev), xo_cpad, out, B, H, W, 32, split)
        _intact("ddnet_upsample4", buf)
        got = out.cpu()
        _exact("ddnet_upsample4", got, want)
    used = set(range(4)) | (set(range(16, 20)) if split else set())
    assert bool((got[..., [k for k in range(32) if k not in used]] == 0).all()), "padded channels must be 0"
    y4, s4 = _y4_64(m.double(), a2.double(), xo4.double(), H, W)
    ref = _up64(y4, H, W)
    Sw = _up64(s4, H, W)
    Mx = s4.amax(dim=(2, 3)).view(3 * B, 1, 4)
    # 6 roundings per term (value, two lerps), the fp32 source coordinate: |d r| <= (2r + 1) 2^-24, slope <= 2 Mx
    ry = torch.arange(H, dtype=torch.float64) * (h2 - 1) / (H - 1)
    rx = torch.arange(W, dtype=torch.float64) * (w2 - 1) / (W - 1)
    dr = ((2 * ry + 2).view(H, 1) + (2 * rx + 2).view(1, W)).reshape(1, H * W, 1)
    eb = U * ((8 + 4 * split) * Sw + 2 * Mx * dr)
    val = got[..., :4].double() + (got[..., 16:20].double() if split else 0)
    _bounded("ddnet_upsample4 B=%d split=%d xo_cpad=%d %dx%d" % (B, split, xo_cpad, H, W), val, ref, eb,
             [("align_corners=False", _up64(y4, H, W, align=False)),
              ("the scalars of slot 0", _up64(_y4_64(m.double(), a2.double(), xo4.double(), H, W, k=0)[0], H, W))])


def r_dd_output(res1, res2, xo2, a3):
    B = res1.shape[0]
    return (a3[:3].view(1, 3, 1) * (res1 + xo2[:B, :, :3].permute(0, 2, 1)) +
            a3[3:].view(1, 3, 1) * (res2 + xo2[B:, :, :3].permute(0, 2, 1)))


def _dd_output64(res1, res2, xo2, a3):
    B = res1.shape[0]
    return (a3[:3].view(1, 3, 1) * (res1 + xo2[:B, :, :3].permute(0, 2, 1)) +
            a3[3:].view(1, 3, 1) * (res2 + xo2[B:, :, :3].permute(0, 2, 1)))


def case_dd_output(dev, B, xo_cpad, H=H_, W=W_):
    g = _gen("dd_output", B, xo_cpad, H, W)
    P = H * W
    res1, res2 = _pos(g, B, 3, P), _pos(g, B, 3, P)
    xo2 = _nan_cols(_pos(g, 2 * B, P, xo_cpad), 3)
    a3 = _pos(g, 6)
    rgb = _pos(g, B, 3, P)
    want, want_m = r_dd_output(res1, res2, xo2, a3), (rgb[:, 0] + rgb[:, 1]) + rgb[:, 2]
    got, got_m = want, want_m
    if dev is not None:
        bo, oo = _dev_out((B, 3, P), dev)
        bm, om = _dev_out((B, P), dev)
        _run("sci_ddnet_output", res1.to(dev), res2.to(dev), xo2.to(dev), xo_cpad, a3.to(dev), oo, B, H, W)
        _run("sci_rgb_sum", rgb.to(dev), om, H, W, B)
        _intact("ddnet_output", bo, bm)
        got, got_m = oo.cpu(), om.cpu()
        _exact("ddnet_output", got, want)
        _exact("rgb_sum", got_m, want_m)
    args = (res1.double(), res2.double(), xo2.double(), a3.double())
    ref = _dd_output64(*args)
    _bounded("ddnet_output B=%d xo_cpad=%d" % (B, xo_cpad), got, ref, 3 * U * ref.abs(),
             [("the two paths' scalars exchanged", _dd_output64(*args[:3], a3.double().roll(3)))])
    r64 = rgb.double()
    _bounded("rgb_sum B=%d" % B, got_m, r64.sum(1), 2 * U * r64.sum(1), [("the blue plane left out", r64[:, :2].sum(1))])


def _site(B, H, W):
    r = torch.arange(H).view(H, 1) & 1
    c = torch.arange(W).view(1, W) & 1
    return (torch.arange(3).view(1, 3, 1, 1) == (r + c).view(1, 1, H, W)).expand(B, 3, H, W)


def case_dd_loss(dev, B, with_dout, H=H_, W=W_):
    g = _gen("dd_loss", B, with_dout, H, W)
    v = _pos(g, B, 3, H, W)
    out = torch.rand(B, 3, H, W, generator=g)
    init = torch.tensor([0.375], dtype=torch.float64)
    site = _site(B, H, W)
    total = B * 3 * H * W
    norm = torch.tensor(2.0) / torch.tensor(float(total))
    x = torch.where(site, out, torch.zeros(()))
    want_d = torch.where(site, norm * (x - v), torch.zeros(()))
    if dev is not None:
        bl, lo = _dev_out((1,), dev, init, torch.float64)
        bd, od = _dev_out((B, 3, H, W), dev) if with_dout else (None, None)
        _run("sci_ddnet_loss_fwd_bwd", v.to(dev), out.to(dev), od, lo, B, H, W)
        _intact("ddnet_loss_fwd_bwd", bl, *([bd] if with_dout else []))
        got_l = lo.cpu()
        got_d = od.cpu() if with_dout else None
        if with_dout:
            _exact("ddnet_loss_fwd_bwd dout", got_d, want_d)
    else:
        d = v - x
        got_l = init + (d * d).double().sum() / total
        got_d = want_d
    out64 = out.double().requires_grad_()
    d64 = v.double() - torch.where(site, out64, torch.zeros((), dtype=torch.float64))
    sq = (d64 * d64).detach()
    loss = (d64 * d64).sum() / total
    ref = init + loss.detach()
    keep = torch.ones(total, dtype=torch.float64)
    keep[(_blocks(total) - 1) * 256:] = 0
    eb = 3 * U * sq.sum() / total + (_blocks(total) + 64) * 2.0 ** -53 * ref
    _bounded("ddnet_loss_fwd_bwd loss B=%d" % B, got_l, ref, eb,
             [("the last ragged block left out", init + (sq.flatten() * keep).sum() / total)])
    if with_dout:
        (gd,) = torch.autograd.grad(loss, out64)
        _bounded("ddnet_loss_fwd_bwd dout B=%d" % B, got_d, gd, 3.01 * U * (2.0 / total) * (out.double().abs() + v.double()) * site,
                 [("the factor 2 left out", gd / 2)])


def case_dd_output_bwd(dev, B, xo_cpad, H=H_, W=W_):
    g = _gen("dd_output_bwd", B, xo_cpad, H, W)
    P = H * W
    dout, res1, res2 = _pos(g, B, 3, P), _pos(g, B, 3, P), _pos(g, B, 3, P)
    xo2 = _nan_cols(_pos(g, 2 * B, P, xo_cpad), 3)
    a3, init = _pos(g, 6), _pos(g, 6)
    d1, d2 = a3[:3].view(1, 3, 1) * dout, a3[3:].view(1, 3, 1) * dout
    want_x = torch.zeros(2 * B, P, 32)
    want_x[:B, :, :3], want_x[B:, :, :3] = d1.permute(0, 2, 1), d2.permute(0, 2, 1)
    if dev is not None:
        bx, ox = _dev_out((2 * B, P, 32), dev)
        b1, o1 = _dev_out((B, 3, P), dev)
        b2, o2 = _dev_out((B, 3, P), dev)
        ba, oa = _dev_out((6,), dev, init)
        _run("sci_ddnet_output_bwd", dout.to(dev), res1.to(dev), res2.to(dev), xo2.to(dev), xo_cpad, a3.to(dev), ox, o1, o2, oa,
             B, H, W)
        _intact("ddnet_output_bwd", bx, b1, b2, ba)
        got_x, got_1, got_2, got_a = ox.cpu(), o1.cpu(), o2.cpu(), oa.cpu()
        _exact("ddnet_output_bwd d_xo2", got_x, want_x)
        _exact("ddnet_output_bwd d_res1", got_1, d1)
        _exact("ddnet_output_bwd d_res2", got_2, d2)
    else:
        got_x, got_1, got_2 = want_x, d1, d2
        got_a = init + torch.cat([(dout * (res1 + xo2[:B, :, :3].permute(0, 2, 1))).sum((0, 2)),
                              (dout * (res2 + xo2[B:, :, :3].permute(0, 2, 1))).sum((0, 2))])
    ins = [res1.double().requires_grad_(), res2.double().requires_grad_(), xo2.double().nan_to_num(0.0).requires_grad_(),
           a3.double().requires_grad_()]
    out = _dd_output64(*ins)

    def grads(gout):
        return torch.autograd.grad(out, ins, gout, retain_graph=True)
    r1, r2, rx, ra = grads(dout.double())
    _exact("ddnet_output_bwd d_res1 vs float64", got_1, r1)
    _exact("ddnet_output_bwd d_res2 vs float64", got_2, r2)
    _exact("ddnet_output_bwd d_xo2 vs float64", got_x[..., :3], rx[..., :3])
    nb = B * _blocks(P)
    dcut = dout.double().clone()
    dcut[B - 1, :, (_blocks(P) - 1) * 256:] = 0
    _bounded("ddnet_output_bwd da3 B=%d xo_cpad=%d" % (B, xo_cpad), got_a, init.double() + ra,
             _sum_bound(init.double() + ra, 2 + TREE + nb + 1),
             [("frame %d's last ragged block left out" % (B - 1), init.double() + grads(dcut)[3])])


def case_dd_mid_bwd(dev, B, path1, H=H_, W=W_):
    g = _gen("dd_mid_bwd", B, path1, H, W)
    P = H * W
    d_t2 = _nan_cols(_pos(g, B, P, 32), 9)
    d_res = _pos(g, B, 3, P)
    m = _pos(g, B, H, W) if path1 else None
    a = _scalars(g, 9)
    init = _pos(g, 9)
    want = torch.zeros(3 * B, P, 32)
    for j in range(3):
        dv = d_t2[..., 3 * j:3 * j + 3]
        want[j * B:(j + 1) * B, :, :3] = dv + d_res.permute(0, 2, 1) if j == 1 else dv
    if dev is not None:
        bx, ox = _dev_out((3 * B, P, 32), dev)
        ba, oa = _dev_out((9,), dev, init) if path1 else (None, None)
        _run("sci_ddnet_stage2_input_bwd", d_t2.to(dev), d_res.to(dev), None if m is None else m.to(dev), ox, oa, B, H, W)
        _intact("ddnet_stage2_input_bwd", bx, *([ba] if path1 else []))
        got_x = ox.cpu()
        got_a = oa.cpu() if path1 else None
        _exact("ddnet_stage2_input_bwd d_xo", got_x, want)
    else:
        got_x = want
        if path1:
            mf = m.reshape(B, P)
            got_a = init.clone()
            for j in range(3):
                got_a[3 * j + 1] += (want[j * B:(j + 1) * B, :, :3].sum(-1) * mf[_src(B, j - 1)]).sum()
    xo64 = torch.zeros(3 * B, P, 3, dtype=torch.float64, requires_grad=True)
    a64 = a.double().requires_grad_()
    m64 = None if m is None else m.double()

    def grads(dt, dr):
        v64, _ = _dd_mid64(m64, a64 if path1 else None, xo64)
        outs = [torch.cat(list(v64), -1), v64[1].permute(0, 2, 1)]
        return torch.autograd.grad(outs, [xo64, a64] if path1 else [xo64], [dt[..., :9], dr], allow_unused=True)
    gr = grads(d_t2.double().nan_to_num(0.0), d_res.double())
    _exact("ddnet_stage2_input_bwd d_xo vs float64", got_x[..., :3], gr[0])
    if path1:
        ref = init.double() + gr[1]
        dt, dr = d_t2.double().nan_to_num(0.0), d_res.double()
        dt[B - 1, (_blocks(P) - 1) * 256:] = 0
        dr[B - 1, :, (_blocks(P) - 1) * 256:] = 0
        _bounded("ddnet_stage2_input_bwd da B=%d" % B, got_a, ref, _sum_bound(ref, 4 + TREE + B * _blocks(P) + 1),
                 [("frame %d's last ragged block left out" % (B - 1), init.double() + grads(dt, dr)[1])])


def case_dd_pack_bwd(dev, B, centre_only, H=H_, W=W_):
    g = _gen("dd_pack_bwd", B, centre_only, H, W)
    P, hp = H * W, (H // 2) * (W // 2)
    m = _pos(g, B, H, W)
    d1 = _nan_cols(_pos(g, 3 * B, P, 32), 3)
    d4 = _nan_cols(_pos(g, 3 * B, hp, 32), 4 if centre_only else 12)
    i1, i4 = _pos(g, 9), _pos(g, 36)
    if dev is not None:
        b1, o1 = _dev_out((9,), dev, i1)
        b4, o4 = _dev_out((36,), dev, i4)
        md = m.to(dev)
        _run("sci_ddnet_pack_input1_bwd", d1.to(dev), md, o1, B, H, W)
        _run("sci_ddnet_pack_input4_bwd", d4.to(dev), md, o4, B, H, W, centre_only)
        _intact("ddnet_pack_input_bwd", b1, b4)
        got1, got4 = o1.cpu(), o4.cpu()
    else:
        got1 = i1 + torch.stack([(d1[j * B:(j + 1) * B, :, k] * m.reshape(B, P)[_src(B, j + k - 2)]).sum()
                                 for j in range(3) for k in range(3)])
        q = _quad(m)
        got4 = i4.clone()
        for j in range(3):
            for k in ((1,) if centre_only else (0, 1, 2)):
                c0 = 0 if centre_only else 4 * k
                got4[(3 * j + k) * 4:(3 * j + k + 1) * 4] += (d4[j * B:(j + 1) * B, :, c0:c0 + 4] * q[_src(B, j + k - 2)]).sum((0, 1))
    a64, a264 = torch.zeros(9, dtype=torch.float64, requires_grad=True), torch.zeros(36, dtype=torch.float64, requires_grad=True)
    m64 = m.double()

    def g1(d):
        return torch.autograd.grad(_dd_pack1_64(m64, a64), a64, d[..., :3])[0]

    def g4(d):
        if centre_only:
            y4, _ = _y4_64(m64, a264, torch.zeros(3 * B, hp, 4, dtype=torch.float64), H, W)
            return torch.autograd.grad(y4, a264, d[..., :4].reshape(3 * B, H // 2, W // 2, 4).permute(0, 3, 1, 2))[0]
        return torch.autograd.grad(_dd_pack4_64(m64, a264), a264, d[..., :12])[0]

    def cut(d, n):
        d = d.clone()
        for j in range(3):
            d[j * B + B - 1, (_blocks(n) - 1) * 256:n] = 0
        return d
    d164, d464 = d1.double().nan_to_num(0.0), d4.double().nan_to_num(0.0)
    ref1, ref4 = i1.double() + g1(d164), i4.double() + g4(d464)
    _bounded("ddnet_pack_input1_bwd B=%d" % B, got1, ref1, _sum_bound(ref1, 1 + TREE + B * _blocks(P) + 1),
             [("frame %d's last ragged block left out" % (B - 1), i1.double() + g1(cut(d164, P)))])
    _bounded("ddnet_pack_input4_bwd B=%d centre_only=%d" % (B, centre_only), got4, ref4,
             _sum_bound(ref4, 1 + TREE + B * _blocks(hp) + 1),
             [("frame %d's last ragged block left out" % (B - 1), i4.double() + g4(cut(d464, hp)))])
    if centre_only:
        other = torch.tensor([(i // 4) % 3 != 1 for i in range(36)])
        assert torch.equal(got4[other], i4[other]), "centre_only must leave the other slots' scalars untouched"


def case_dd_up4_bwd(dev, B, H=H_, W=W_):
    g = _gen("dd_up4_bwd", B, H, W)
    P, h2, w2 = H * W, H // 2, W // 2
    hp, n = h2 * w2, 3 * B
    d_up = _nan_cols(_pos(g, n, P, 32), 4)
    init = _pos(g, n, hp, 32)
    if dev is not None:
        buf, out = _dev_out((n, hp, 32), dev, init)
        _run("sci_ddnet_upsample4_bwd", d_up.to(dev), out, B, H, W)
        _intact("ddnet_upsample4_bwd", buf)
        got = out.cpu()
    else:
        y0, y1, ly0, ly1 = _up_coords(H, h2)
        x0, x1, lx0, lx1 = _up_coords(W, w2)
        got = init.clone()
        gv = d_up[..., :4].reshape(n, H, W, 4)
        for yy, ly in ((y0, ly0), (y1, ly1)):
            for xx, lx in ((x0, lx0), (x1, lx1)):
                c = (ly.view(H, 1) * lx.view(1, W)).view(1, H, W, 1) * gv
                idx = (yy.view(H, 1) * w2 + xx.view(1, W)).reshape(-1)
                got[..., :4].index_add_(1, idx, c.reshape(n, P, 4))
    assert torch.equal(got[..., 4:], init[..., 4:]), "channels 4.. of d_y4 must stay untouched"
    y4 = torch.zeros(n, 4, h2, w2, dtype=torch.float64, requires_grad=True)
    up = F.interpolate(y4, size=(H, W), mode="bilinear", align_corners=True)

    def adj(d):
        return torch.autograd.grad(up, y4, d[..., :4].reshape(n, H, W, 4).permute(0, 3, 1, 2), retain_graph=True)[0] \
            .permute(0, 2, 3, 1).reshape(n, hp, 4)
    d64 = d_up.double().nan_to_num(0.0)
    ref = init[..., :4].double() + adj(d64)

    # every target collects from the full-resolution pixels whose source cell lies within one row / column of it
    def near(n_, n2):
        r0 = torch.floor(torch.arange(n_, dtype=torch.float64) * (n2 - 1) / (n_ - 1)).long()
        R = torch.zeros(n_, n2, dtype=torch.float64)
        for d in (-1, 0, 1, 2):
            R[torch.arange(n_), (r0 + d).clamp(0, n2 - 1)] = 1
        return R
    Ry, Rx = near(H, h2), near(W, w2)
    G = torch.einsum("yi,nyxc,xj->nijc", Ry, d64[..., :4].reshape(n, H, W, 4).abs(), Rx).reshape(n, hp, 4)
    cnt = 4 * torch.einsum("yi,xj->ij", Ry, Rx).reshape(1, hp, 1)
    dn = 2 * (h2 - 1) + 2 * (w2 - 1) + 6
    eb = U * ((cnt + 1) * (init[..., :4].double() + G) + dn * G)
    cutd = d64.clone()
    cutd[n - 1, (_blocks(P) - 1) * 256:] = 0
    _bounded("ddnet_upsample4_bwd B=%d %dx%d" % (B, H, W), got[..., :4], ref, eb,
             [("the last ragged block of the last image left out", init[..., :4].double() + adj(cutd))])


# ---- training bookkeeping --------------------------------------------------------------------------------------------
def case_act_bwd(dev, C, relu, y_null, sums):
    g = _gen("act_bwd", C, relu, y_null, sums)
    rows, grid = max(1, 256 // C), 148 * 8
    n_pix = grid * rows * 3 // 2 + 1                   # a second grid-stride pass over a third of the pixels
    dy = _pos(g, n_pix, C)
    y = _pos(g, n_pix, C)
    if relu:
        r = torch.rand(n_pix, C, generator=g)
        y = torch.where(r < 0.25, -y, torch.where(r < 0.3, torch.zeros(()), y))
    yk = None if y_null else y
    i1, i2 = _pos(g, C), _pos(g, C)
    want = torch.where(~(y > 0), torch.zeros(()), dy) if relu else dy.clone()
    s_on = (sums, sums and not y_null)
    if dev is not None:
        bz, oz = _dev_out((n_pix, C), dev)
        b1, o1 = _dev_out((C,), dev, i1) if s_on[0] else (None, None)
        b2, o2 = _dev_out((C,), dev, i2) if s_on[1] else (None, None)
        _run("sci_act_bwd", dy.to(dev), None if yk is None else yk.to(dev), oz, n_pix, C, relu, o1, o2)
        _intact("act_bwd", bz, *[b for b in (b1, b2) if b is not None])
        got = oz.cpu()
        _exact("act_bwd dz", got, want)
        got1 = o1.cpu() if s_on[0] else None
        got2 = o2.cpu() if s_on[1] else None
    else:
        got = want
        got1, got2 = i1 + want.sum(0), i2 + (want * y).sum(0)
    y64 = y.double().requires_grad_()
    (dz,) = torch.autograd.grad(F.relu(y64) if relu else y64, y64, dy.double())
    _bounded("act_bwd dz C=%d relu=%d" % (C, relu), got, dz, 0.0)
    depth = _blocks(n_pix, grid * rows) + rows + grid + 2
    keep = torch.zeros(n_pix, 1, dtype=torch.float64)
    keep[:grid * rows] = 1
    tag = "act_bwd C=%d relu=%d" % (C, relu)
    if s_on[0]:
        ref = i1.double() + dz.sum(0)
        _bounded(tag + " s1", got1, ref, _sum_bound(ref, depth), [("the second pass left out", i1.double() + (dz * keep).sum(0))])
    if s_on[1]:
        t = dz * y.double()
        ref = i2.double() + t.sum(0)
        _bounded(tag + " s2", got2, ref, _sum_bound(ref, depth + 1), [("the second pass left out", i2.double() + (t * keep).sum(0))])


def case_meas_loss(dev, C, strip, with_dx, B=3, H=H_, W=W_):
    g = _gen("meas_loss", C, strip, with_dx, B, H, W)
    P = H * W
    xhat = _pos(g, B, C, H, W)
    phi = _pos(g, B, H, W)
    y = torch.rand(H, W, generator=g) * B
    init = torch.tensor([0.625], dtype=torch.float64)
    norm_pixels = 3 * P if strip else 0
    cnt = float(norm_pixels or P)
    ch = (_site(1, H, W)[0].float().argmax(0) if C == 3 else torch.zeros(H, W, dtype=torch.long))
    pick = xhat.gather(1, ch.expand(B, 1, H, W)).squeeze(1)            # [B][H][W]: the sampled channel
    up = torch.zeros(H, W)
    for t in range(B):
        up = up + pick[t] * phi[t]
    diff = up - y
    gsc = torch.tensor(2.0 / cnt, dtype=torch.float32) * diff
    want = torch.zeros(B, C, H, W)
    for t in range(B):
        want[t].scatter_(0, ch[None], (gsc * phi[t])[None])
    if dev is not None:
        bl, lo = _dev_out((1,), dev, init, torch.float64)
        bd, od = _dev_out((B, C, H, W), dev) if with_dx else (None, None)
        _run("sci_meas_loss_fwd_bwd", xhat.to(dev), phi.to(dev), y.to(dev), od, lo, H, W, B, C, norm_pixels)
        _intact("meas_loss", bl, *([bd] if with_dx else []))
        got_l = lo.cpu()
        got_d = od.cpu() if with_dx else None
        if with_dx:
            _exact("meas_loss_fwd_bwd dxhat", got_d, want)
    else:
        got_l, got_d = init + (diff.double() ** 2).sum() / cnt, want
    x64 = xhat.double().requires_grad_()
    up64 = (x64.gather(1, ch.expand(B, 1, H, W)).squeeze(1) * phi.double()).sum(0)
    d64 = up64 - y.double()
    loss = (d64 * d64).sum() / cnt
    ref = init + loss.detach()
    S_up = (pick.double() * phi.double()).sum(0)
    e_d = U * (2 * B * S_up + S_up + y.double())                     # the fp32 sum over frames, then the difference
    dd = d64.detach().abs()
    eb_px = 2 * dd * e_d + e_d * e_d + U * dd * dd
    keep = torch.ones(P, dtype=torch.float64)
    keep[(_blocks(P) - 1) * 256:] = 0
    sq = (d64.detach() ** 2).flatten()
    _bounded("meas_loss C=%d strip=%d" % (C, strip), got_l, ref, eb_px.sum() / cnt + (_blocks(P) + 64) * 2.0 ** -53 * ref,
             [("the last ragged block left out", init + (sq * keep).sum() / cnt)])
    if with_dx:
        (gd,) = torch.autograd.grad(loss, x64)
        eb = (2.0 / cnt) * (e_d * phi.double()).unsqueeze(1) * (gd != 0) + 3.01 * U * gd.abs()
        _bounded("meas_loss dxhat C=%d strip=%d" % (C, strip), got_d, gd, eb, [("the factor 2 left out", gd / 2)])


# ---- sci_ops.cu bookkeeping ------------------------------------------------------------------------------------------
def case_dual_stage1(dev, first, B=2, H=6, W=600):
    """W / 2 = 300 threads a row: a full block of 256 and a ragged one of 44."""
    g = _gen("dual_stage1", first, B, H, W)
    xhat = 1.4 * torch.rand(B, 3, H, W, generator=g) - 0.2
    x, b, orig = torch.rand(B, H, W, generator=g), torch.rand(B, H, W, generator=g) - 0.5, torch.rand(B, H, W, generator=g)
    init = torch.tensor([1.5], dtype=torch.float64)
    site = _site(B, H, W)
    s = (xhat * site).sum(1)                                   # exact: one nonzero term
    t = torch.clamp(s, 0.0, 1.0)
    xv = s if first else x
    want_b = b - (xv - t)
    if dev is not None:
        bx, ox = _dev_out((B, H, W), dev, x)
        bb, ob = _dev_out((B, H, W), dev, b)
        bt, ot = _dev_out((B, H, W), dev)
        bs, os_ = _dev_out((1,), dev, init, torch.float64)
        _run("sci_dual_update_stage1", xhat.to(dev), ox, ob, ot, first, H, W, B, orig.to(dev), os_)
        _intact("dual_update_stage1", bx, bb, bt, bs)
        got_x, got_b, got_t, got_s = ox.cpu(), ob.cpu(), ot.cpu(), os_.cpu()
        _exact("dual_update_stage1 x", got_x, xv)
        _exact("dual_update_stage1 b", got_b, want_b)
        _exact("dual_update_stage1 theta", got_t, t)
    else:
        got_x, got_b, got_t = xv, want_b, t
        got_s = init + ((xv - orig) ** 2).double().sum()
    x64 = xhat.double()
    ts = torch.where(site, x64, torch.zeros((), dtype=torch.float64)).sum(1)
    bad = torch.where(site.flip(1), x64, torch.zeros((), dtype=torch.float64)).sum(1)
    _bounded("dual_update_stage1 theta", got_t, ts.clamp(0, 1), 0.0, [("the wrong CFA sites", bad.clamp(0, 1))])
    xr = ts if first else x.double()
    _bounded("dual_update_stage1 x", got_x, xr, 0.0)
    refb = b.double() - (xr - ts.clamp(0, 1))
    _bounded("dual_update_stage1 b first=%d" % first, got_b, refb, 2 * U * (b.double().abs() + xr.abs() + 1),
             [("the wrong CFA sites", b.double() - (xr - bad.clamp(0, 1)))])
    sq = (xr - orig.double()) ** 2
    keep = torch.ones(B, H, W, dtype=torch.float64)
    keep[B - 1, H - 1, 512:] = 0
    ref = init + sq.sum()
    _bounded("dual_update_stage1 sse first=%d" % first, got_s, ref, 3 * U * sq.sum() + (B * H * 2 + 64) * 2.0 ** -53 * ref,
             [("the last ragged block left out", init + (sq * keep).sum())])


def case_dual_gray(dev, first, n=3 * 2660 + 5):
    g = _gen("dual_gray", first, n)
    xhat = 1.4 * torch.rand(n, generator=g) - 0.2
    x_pre, w, x, b, orig = (torch.rand(n, generator=g) for _ in range(5))
    init = torch.tensor([0.5], dtype=torch.float64)
    th = torch.clamp(xhat, 0.0, 1.0)
    want_w = w + (x_pre - xhat)
    want_b = b + ((xhat if first else x) - th)
    if dev is not None:
        bw, ow = _dev_out((n,), dev, w)
        bb, ob = _dev_out((n,), dev, b)
        bt, ot = _dev_out((n,), dev)
        bs, os_ = _dev_out((1,), dev, init, torch.float64)
        _run("sci_dual_update_gray", xhat.to(dev), x_pre.to(dev), ow, x.to(dev), ob, ot, first, n, orig.to(dev), os_)
        _intact("dual_update_gray", bw, bb, bt, bs)
        got_w, got_b, got_t, got_s = ow.cpu(), ob.cpu(), ot.cpu(), os_.cpu()
        _exact("dual_update_gray w", got_w, want_w)
        _exact("dual_update_gray b", got_b, want_b)
        _exact("dual_update_gray theta", got_t, th)
    else:
        got_w, got_b, got_t = want_w, want_b, th
        got_s = init + ((th - orig) ** 2).double().sum()
    xh, xp = xhat.double(), x_pre.double()
    t64 = xh.clamp(0, 1)
    _bounded("dual_update_gray theta", got_t, t64, 0.0)
    _bounded("dual_update_gray w", got_w, w.double() + (xp - xh), 2 * U * (w.double() + xp + xh.abs()),
             [("the sign of the step", w.double() - (xp - xh))])
    xv = xh if first else x.double()
    _bounded("dual_update_gray b first=%d" % first, got_b, b.double() + (xv - t64), 2 * U * (b.double() + xv.abs() + t64),
             [("the unclipped theta", b.double() + (xv - xh))])
    sq = (t64 - orig.double()) ** 2
    ref = init + sq.sum()
    _bounded("dual_update_gray sse", got_s, ref, 3 * U * sq.sum() + (_blocks(n) + 64) * 2.0 ** -53 * ref,
             [("the last ragged block left out", init + sq[:(_blocks(n) - 1) * 256].sum())])


def case_closed_form(dev, clip, B=2, H=6, W=300):
    g = _gen("closed_form", clip, B, H, W)
    x, b = torch.rand(B, H, W, generator=g), torch.rand(B, H, W, generator=g) - 0.5
    xhat, w = 1.4 * torch.rand(B, 3, H, W, generator=g) - 0.2, 0.2 * torch.rand(B, 3, H, W, generator=g) - 0.1
    rho, tau = 0.3, 0.7
    inv_tau = float(torch.tensor(1.0) / torch.tensor(tau))
    site = _site(B, H, W)
    m = site.float()
    num = torch.tensor(rho) * (m * x[:, None])
    num = num + m * b[:, None]
    num = num + torch.tensor(tau) * xhat
    num = num + w
    v = num / (torch.tensor(rho) * m + torch.tensor(tau))
    if clip:
        v = torch.clamp(v, 0.0, 1.0)
    want_u = v - torch.tensor(inv_tau) * w
    if dev is not None:
        bx, ox = _dev_out((B, 3, H, W), dev)
        bu, ou = _dev_out((B, 3, H, W), dev)
        _run("sci_closed_form_demosaic", x.to(dev), b.to(dev), xhat.to(dev), w.to(dev), rho, tau, inv_tau, clip, ox, ou, H, W, B)
        _intact("closed_form_demosaic", bx, bu)
        got_x, got_u = ox.cpu(), ou.cpu()
        _exact("closed_form_demosaic x_rgb", got_x, v)
        _exact("closed_form_demosaic u", got_u, want_u)
    else:
        got_x, got_u = v, want_u
    rho64, tau64, it64 = (float(torch.tensor(s)) for s in (rho, tau, inv_tau))

    def ref_of(mm):
        mm = mm.double()
        nm = rho64 * mm * x.double()[:, None] + mm * b.double()[:, None] + tau64 * xhat.double() + w.double()
        den = rho64 * mm + tau64
        S = (rho64 * mm * x.double()[:, None]).abs() + (mm * b.double()[:, None]).abs() + tau64 * xhat.double().abs() + w.double().abs()
        r = nm / den
        return (r.clamp(0, 1) if clip else r), S / den
    ref, Sd = ref_of(site)
    bad, _ = ref_of(site.flip(1))
    ebx = U * (4.1 * Sd + 2.1 * ref.abs())
    tag = "closed_form_demosaic clip=%d" % clip
    _bounded(tag + " x_rgb", got_x, ref, ebx, [("the wrong CFA sites", bad)])
    _bounded(tag + " u", got_u, ref - it64 * w.double(), ebx + 2.1 * U * (ref.abs() + (it64 * w.double()).abs()),
             [("the wrong CFA sites", bad - it64 * w.double())])


def case_pad_crop(dev, kind, planes, H, W, Ho, Wo):
    g = _gen("pad", kind, planes, H, W, Ho, Wo)
    x = torch.rand(planes, H, W, generator=g)
    if kind == "crop":
        ref = x.double()[:, :Ho, :Wo]
        bad = x.double()[:, H - Ho:, W - Wo:]
    else:
        mode = "reflect" if kind == "reflect" else "replicate"
        ref = F.pad(x.double()[None], (0, Wo - W, 0, Ho - H), mode=mode)[0]
        bad = F.pad(x.double()[None], (0, Wo - W, 0, Ho - H), mode="replicate" if kind == "reflect" else "constant")[0]
    got = ref.float()
    if dev is not None:
        buf, out = _dev_out((planes, Ho, Wo), dev)
        _run({"reflect": "sci_reflect_pad2d", "replicate": "sci_replicate_pad2d", "crop": "sci_crop2d"}[kind], x.to(dev), out,
             planes, H, W, Ho, Wo)
        _intact(kind, buf)
        got = out.cpu()
    teeth = [] if torch.equal(bad, ref) else [("the other border rule", bad)]
    _bounded("%s %dx%d -> %dx%d" % (kind, H, W, Ho, Wo), got, ref, 0.0, teeth)


def case_axpy(dev, n=2660 + 3):
    g = _gen("axpy", n)
    x, y = torch.rand(n, generator=g), torch.rand(n, generator=g) - 0.5
    a = -0.3
    want = x + torch.tensor(a) * y
    got = want
    if dev is not None:
        buf, out = _dev_out((n,), dev)
        _run("sci_axpy", x.to(dev), a, y.to(dev), out, n)
        _intact("axpy", buf)
        got = out.cpu()
        _exact("axpy", got, want)
    a64 = float(torch.tensor(a))
    ref = x.double() + a64 * y.double()
    _bounded("axpy", got, ref, 2 * U * (x.double() + abs(a64) * y.double().abs()),
             [("the sign of a", x.double() - a64 * y.double())])


# ---- GPU cases -------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("C,rnd,Cpad", [(1, 0, 5), (3, 0, 13), (1, 1, 32), (3, 1, 32), (3, 0, 48), (1, 1, 48)])
def test_ffdnet_pack_input(cuda, C, rnd, Cpad):
    case_ffdnet_pack(cuda, C, rnd, Cpad)


@gpu
def test_ffdnet_pack_input_edges(cuda):
    case_ffdnet_pack(cuda, 3, 1, 32, B=1, H=4, W=4)          # 2x2 at half resolution
    case_ffdnet_pack(cuda, 1, 0, 5, B=3, H=6, W=66)          # half-resolution width 33


@gpu
@pytest.mark.parametrize("C,Cpad", [(1, 4), (3, 12), (3, 32), (1, 48)])
def test_ffdnet_unpack_output(cuda, C, Cpad):
    case_ffdnet_unpack(cuda, C, Cpad)


@gpu
@pytest.mark.parametrize("C", [1, 3])
def test_ffdnet_split_half(cuda, C):
    case_ffdnet_split_half(cuda, C)
    case_ffdnet_split_half(cuda, C, B=1, H=4, W=4)


@gpu
@pytest.mark.parametrize("Cpad,rnd,B", [(12, 0, 1), (16, 0, 2), (32, 0, 7), (48, 0, 3), (32, 1, 3), (48, 1, 2)])
def test_fastdvd_pack_input(cuda, Cpad, rnd, B):
    case_fdvd_pack(cuda, Cpad, rnd, B)


@gpu
def test_fastdvd_pack_input_edges(cuda):
    case_fdvd_pack(cuda, 48, 1, 1, H=2, W=2)
    case_fdvd_pack(cuda, 12, 0, 3, H=6, W=66)


@gpu
@pytest.mark.parametrize("C,B", [(32, 3), (64, 2), (64, 1)])
def test_fastdvd_pack_input_half(cuda, C, B):
    case_fdvd_half(cuda, C, B)


@gpu
@pytest.mark.parametrize("B,acc", [(1, 1), (2, 0), (3, 1), (7, 0)])
def test_fastdvd_pack_input_grad(cuda, B, acc):
    case_fdvd_pack_grad(cuda, B, acc)


@gpu
@pytest.mark.parametrize("Cpad,B", [(3, 2), (32, 3), (48, 1), (64, 7)])
def test_fastdvd_output_and_grad(cuda, Cpad, B):
    case_fdvd_output(cuda, Cpad, B)


@gpu
def test_fastdvd_noisy_input(cuda):
    case_fdvd_noisy(cuda)


@gpu
@pytest.mark.parametrize("B,split", [(1, 1), (2, 0), (3, 1), (7, 0)])
def test_ddnet_pack_input(cuda, B, split):
    case_dd_pack(cuda, B, split)


@gpu
@pytest.mark.parametrize("B,split,xo_cpad,path1", [(1, 0, 3, True), (2, 1, 32, True), (7, 1, 64, True), (3, 1, 3, False),
                                                   (2, 0, 64, False)])
def test_ddnet_stage2_input(cuda, B, split, xo_cpad, path1):
    case_dd_mid(cuda, B, split, xo_cpad, path1)


@gpu
@pytest.mark.parametrize("B,split,xo_cpad,H,W", [(2, 0, 4, H_, W_), (3, 1, 32, H_, W_), (7, 0, 64, H_, W_), (1, 1, 4, 4, 4),
                                                 (2, 0, 32, 4, 10)])
def test_ddnet_upsample4(cuda, B, split, xo_cpad, H, W):
    case_dd_up4(cuda, B, split, xo_cpad, H, W)


@gpu
@pytest.mark.parametrize("B,xo_cpad", [(1, 3), (3, 32), (7, 64)])
def test_ddnet_output_and_rgb_sum(cuda, B, xo_cpad):
    case_dd_output(cuda, B, xo_cpad)


@gpu
@pytest.mark.parametrize("B,with_dout", [(2, True), (3, False)])
def test_ddnet_loss_fwd_bwd(cuda, B, with_dout):
    case_dd_loss(cuda, B, with_dout)


@gpu
@pytest.mark.parametrize("B,xo_cpad", [(1, 3), (2, 32), (7, 64)])
def test_ddnet_output_bwd(cuda, B, xo_cpad):
    case_dd_output_bwd(cuda, B, xo_cpad)


@gpu
@pytest.mark.parametrize("B,path1", [(1, True), (3, True), (7, True), (2, False)])
def test_ddnet_stage2_input_bwd(cuda, B, path1):
    case_dd_mid_bwd(cuda, B, path1)


@gpu
@pytest.mark.parametrize("B,centre_only", [(1, 0), (2, 1), (3, 0), (7, 1)])
def test_ddnet_pack_input_bwd(cuda, B, centre_only):
    case_dd_pack_bwd(cuda, B, centre_only)


@gpu
@pytest.mark.parametrize("B,H,W", [(2, H_, W_), (7, H_, W_), (1, 4, 4), (3, 4, 10)])
def test_ddnet_upsample4_bwd(cuda, B, H, W):
    case_dd_up4_bwd(cuda, B, H, W)


@gpu
@pytest.mark.parametrize("C,relu,y_null,sums", [(3, 1, False, True), (32, 0, False, True), (48, 1, False, True),
                                                (96, 0, True, True), (128, 1, False, False)])
def test_act_bwd(cuda, C, relu, y_null, sums):
    case_act_bwd(cuda, C, relu, y_null, sums)


@gpu
@pytest.mark.parametrize("C,strip,with_dx", [(1, False, True), (3, True, True), (3, False, False)])
def test_meas_loss_fwd_bwd(cuda, C, strip, with_dx):
    case_meas_loss(cuda, C, strip, with_dx)


@gpu
@pytest.mark.parametrize("first", [0, 1])
def test_dual_update_stage1(cuda, first):
    case_dual_stage1(cuda, first)


@gpu
@pytest.mark.parametrize("first", [0, 1])
def test_dual_update_gray(cuda, first):
    case_dual_gray(cuda, first)


@gpu
@pytest.mark.parametrize("clip", [0, 1])
def test_closed_form_demosaic(cuda, clip):
    case_closed_form(cuda, clip)


@gpu
@pytest.mark.parametrize("kind,H,W,Ho,Wo", [("reflect", 5, 7, 9, 13), ("reflect", 1, 6, 1, 8), ("replicate", 5, 7, 8, 12),
                                            ("replicate", 1, 1, 3, 4), ("crop", 9, 13, 5, 7), ("crop", 5, 7, 1, 7)])
def test_pad_crop(cuda, kind, H, W, Ho, Wo):
    case_pad_crop(cuda, kind, 3, H, W, Ho, Wo)


@gpu
def test_axpy(cuda):
    case_axpy(cuda)


# ---- CPU only: every float32 restatement against its float64 statement, with the same bounds and teeth ---------------
CPU_CASES = [
    (case_ffdnet_pack, (1, 1, 32)), (case_ffdnet_pack, (3, 0, 13)), (case_ffdnet_unpack, (3, 12)), (case_ffdnet_split_half, (3,)),
    (case_fdvd_pack, (32, 1, 3)), (case_fdvd_pack, (12, 0, 2)), (case_fdvd_half, (64, 2)), (case_fdvd_pack_grad, (3, 1)),
    (case_fdvd_output, (32, 3)), (case_fdvd_noisy, ()), (case_dd_pack, (3, 1)), (case_dd_mid, (2, 1, 32, True)),
    (case_dd_mid, (3, 1, 3, False)), (case_dd_up4, (3, 1, 32)), (case_dd_up4, (2, 0, 4, 4, 10)), (case_dd_output, (2, 32)),
    (case_dd_loss, (2, True)), (case_dd_output_bwd, (2, 32)), (case_dd_mid_bwd, (3, True)), (case_dd_pack_bwd, (3, 0)),
    (case_dd_pack_bwd, (2, 1)), (case_dd_up4_bwd, (2,)), (case_dd_up4_bwd, (1, 4, 4)), (case_act_bwd, (48, 1, False, True)),
    (case_meas_loss, (3, True, True)), (case_dual_stage1, (1,)), (case_dual_gray, (0,)), (case_closed_form, (1,)),
    (case_pad_crop, ("reflect", 3, 5, 7, 9, 13)), (case_axpy, ()),
]


@pytest.mark.parametrize("fn,args", CPU_CASES, ids=["%s%s" % (f.__name__[5:], a) for f, a in CPU_CASES])
def test_restatements_against_float64_cpu(fn, args):
    fn(None, *args)
