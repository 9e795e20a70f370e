"""Tensor-core convolution, per launch plan, against float64.

Every kernel plan of ``sci_conv3x3_fwd`` / ``_dgrad`` / ``_wgrad`` the planner can pick (forced through its environment
knobs, and confirmed from the plan line it prints under ``SCI_CONV_VERBOSE=1``) runs at ragged sizes - rows spanning three
128-pixel tiles with a short last one, heights that are not a multiple of the rows per super-tile - and is compared element
by element with a float64 reference of the same operation.

Operands are first rounded to the format the path multiplies (TF32 round-to-nearest-away, or fp16), so every product is
exact in fp32 and what remains is accumulation plus the epilogue.  Per element the error must stay within

    |got - ref| <= C_ACC * K * 2^-24 * S  (+ epilogue roundings, + half an ulp of the stored format)

with S the float64 convolution of |x| with |w| (the sum of |terms|) and K the number of products summed.  Each addition of
an fp32 accumulation chain errs by at most one ulp of its partial sum (2^-23 relative if the tensor core's internal adder
truncates), and every partial sum is at most S, so C_ACC = 2 holds whatever the adder's rounding.  The split forms (fp32
value + remainder, fp16 value + remainder x 2^11) are compared with the UNquantised fp32 operands instead: SPLIT_REL * S for
the representation plus the same accumulation term per accumulator chain (_split_bound).  With split accumulators the
value x value chain is the only long one; in ONE accumulator the small products lengthen it, which is what the split
accumulators avoid.

Each case also checks that the bound has teeth: a reference with one 8-channel K slice of one tap missing at the last pixel
of the last (ragged) tile must violate it, and for split forms so must the reference with either cross product (value x
weight remainder, activation remainder x value) left out on its own.  Outputs are prefilled
with NaN inside a larger allocation whose margins hold a sentinel: every valid element must be finite and every margin
untouched.  Every case prints max and RMS of err / bound (run pytest with -s to see them)."""
import ctypes
import math
import os
import re
import zlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

C_ACC = 2.0
# Split forms: with x = xh + xl + ex (xh the leading part, xl the rounded remainder) and |ex| <= 2^-22 |x| (TF32 RNA:
# |x - xh| <= 2^-11 |x|, and rounding that remainder to 11 bits errs by 2^-11 of it; fp16 value + fp16(remainder x 2^11)
# likewise), the three products xh wh + xh wl + xl wh differ from x w by xl wl + ex w' + x' ew + ex ew
# <= 3 * 2^-22 * (1 + 2^-10) |x w| < 2^-20 |x w|.
SPLIT_REL = 2.0 ** -20
SENTINEL = -7.75                      # exact in fp32 and fp16
MARGIN = 1024                         # elements before and after every output (keeps TMA base addresses 2 KB aligned)
N_, H_, W_ = 2, 37, 300               # W: tiles of 128 + 128 + 44 pixels; H: no multiple of 2, 4 or 8
SCI_EUNSUPPORTED = -3
KNOBS = ("SCI_CONV_V2", "SCI_CONV_RESIDENT", "SCI_CONV_WPAIR", "SCI_CONV_ROWS", "SCI_CONV_STACK", "SCI_CONV_EPI_WG",
         "SCI_CONV_TPS", "SCI_CONV_SPLIT_ACC", "SCI_CONV_PDL", "SCI_WGRAD_V3", "SCI_CONV_SW64", "SCI_CONV_IMPL",
         "SCI_FFDNET_INF", "SCI_CONV_HALF")


@pytest.fixture(autouse=True)
def _plan_env(monkeypatch):
    """Every case starts from the planner's defaults and prints its launch plans."""
    assert "SCI_CONV_DBG" not in os.environ, "SCI_CONV_DBG is a timing experiment (results invalid): unset it"
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("SCI_CONV_VERBOSE", "1")


# ---- rounding ------------------------------------------------------------------------------------------------------
def tf32(t):
    """cvt.rna.tf32.f32: round to 10 explicit mantissa bits, ties away from zero (the carry of +0x1000 does that)."""
    i = t.contiguous().view(torch.int32)
    return ((i + 0x1000) & -8192).view(torch.float32)


def half_split(v):
    """fp16 value + fp16 remainder x 2^11 of fp32 values."""
    hv = v.half()
    return hv, ((v - hv.float()) * 2048.0).half()


# ---- plumbing ------------------------------------------------------------------------------------------------------
def coherent(shape, scale, quant, g, dev):
    """Operands of the split-form cases: positive values scale * 2^U(-1,1) whose rounded part (`quant`: TF32 or fp16, 10
    explicit mantissa bits) has a mantissa in [1, 1.25) and whose remainder is 0.3 to 0.45 of its ulp, i.e. 2.4e-4 to
    4.4e-4 of the value.  Every product the split forms add back (value x remainder, remainder x value) is then positive
    and at least 2.4e-4 of its term: none of them can cancel, so leaving out either one moves every convolution sum by more than
    2^-12.4 of its S, which the split-form bound (see _split_bound) cannot absorb."""
    def r():
        return torch.rand(shape, generator=g).to(dev)
    _, e = torch.frexp(scale * torch.exp2(2 * r() - 1))
    hi = quant(torch.ldexp(0.5 + 0.125 * r(), e))
    _, eh = torch.frexp(hi)
    out = hi + (0.3 + 0.15 * r()) * torch.ldexp(torch.ones_like(hi), eh - 11)
    assert bool((quant(out) == hi).all())
    return out


def _lib():
    from adaptivepnp_sci_b200 import _lib
    return _lib


def _desc(**kw):
    from adaptivepnp_sci_b200 import engine
    d = engine.ConvDesc()
    for k, v in kw.items():
        setattr(d, k, v.data_ptr() if isinstance(v, torch.Tensor) else v)
    return d


def _launch(d, impl=0):
    L = _lib()
    return L.lib.sci_conv3x3_fwd(ctypes.byref(d), impl, L.stream())


def _guarded(shape, dtype, dev):
    n = int(np.prod(shape))
    buf = torch.full((n + 2 * MARGIN,), SENTINEL, dtype=dtype, device=dev)
    t = buf[MARGIN:MARGIN + n].view(shape)
    t.fill_(float("nan"))
    return buf, t


def _margins_intact(buf):
    return bool((buf[:MARGIN] == SENTINEL).all()) and bool((buf[-MARGIN:] == SENTINEL).all())


def _bits(t):
    return t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32)


def _plans(capfd, prefix):
    """Key/value fields of every plan line with this prefix printed since the last call."""
    out = []
    for line in capfd.readouterr().err.splitlines():
        if not line.startswith(prefix):
            continue
        toks = line[len(prefix):].replace("|", " ").split()
        f = {}
        for a, b in zip(toks, toks[1:]):
            if re.fullmatch(r"-?\d+", b):
                f.setdefault(a, int(b))
            elif re.fullmatch(r"\d+/\d+", b):
                f.setdefault(a, b)
        m = re.search(r"\(\+(\d+)\)", line)
        if m:
            f["col0"] = int(m.group(1))
        out.append(f)
    return out


def _assert_plan(plans, want, n=1):
    assert len(plans) == n, "expected %d plan line(s), got %s" % (n, plans)
    for p in plans:
        bad = {k: (p.get(k), v) for k, v in want.items() if p.get(k) != v}
        assert not bad, "plan %s: (got, wanted) %s" % (p, bad)


def _report(tag, err, bound):
    r = (err / bound).flatten()
    mx, rms = float(r.max()), float(torch.sqrt((r * r).mean()))
    print("[%s] max(err/bound) %.3g  rms(err/bound) %.3g" % (tag, mx, rms))
    return mx


def _ref_conv(x64, w64, stride):
    """x [N,H,W,K], packed w [9,Cout,K] (tap = 3 r + s) -> [N,Ho,Wo,Cout] in float64, 32 rows at a time."""
    Cout, K = w64.shape[1], w64.shape[2]
    wt = w64.view(3, 3, Cout, K).permute(2, 3, 0, 1).contiguous()
    xt = x64.permute(0, 3, 1, 2)
    H = xt.shape[2]
    Ho = (H - 1) // stride + 1
    outs = []
    rows = 32
    for r0 in range(0, Ho, rows):
        r1 = min(Ho, r0 + rows)
        lo, hi = r0 * stride - 1, (r1 - 1) * stride + 2          # input rows that output rows [r0, r1) read
        xs = xt[:, :, max(lo, 0):min(hi, H)]
        xs = F.pad(xs, (0, 0, max(0, -lo), max(0, hi - H)))
        outs.append(F.conv2d(xs, wt, stride=stride, padding=(0, 1)))
    return torch.cat(outs, 2).permute(0, 2, 3, 1)


def _pix_shuffle(t, ps):
    """GEMM column q * (C/4) + c -> sub-pixel q = dy * 2 + dx, channel c (NHWC)."""
    if not ps:
        return t
    N, H, W, C = t.shape
    return t.view(N, H, W, 2, 2, C // 4).permute(0, 1, 3, 2, 4, 5).reshape(N, 2 * H, 2 * W, C // 4)


# ---- forward / data-gradient cases ---------------------------------------------------------------------------------
# form: tf32 (fp32 path, TF32 operands) | wsplit (fp32 path, value + remainder weights) | lo (3xTF32: input written with
# emit_lo, weights duplicated over both halves, split accumulators via lo_channel0) | f16 | hsplit (fp16 value + remainder)
def _case(cid, Cin, Cout, plan, kernel="v2", form="tf32", env=None, N=N_, H=H_, W=W_, stride=1, relu=1, affine=True, ps=0,
          res=False, round_tf32=0, emit_lo=0, k_used=0, cin_store=0, cout_store=0, planar=False, mask=None, n_plans=1,
          fill=False):
    return pytest.param(dict(Cin=Cin, Cout=Cout, plan=plan, kernel=kernel, form=form, env=env or {}, N=N, H=H, W=W,
                             stride=stride, relu=relu, affine=affine, ps=ps, res=res, round_tf32=round_tf32, emit_lo=emit_lo,
                             k_used=k_used, cin_store=cin_store, cout_store=cout_store, planar=planar, mask=mask,
                             n_plans=n_plans, fill=fill), id=cid)


V2F = dict(half=0, rb="128/128")
FWD_CASES = [
    # row-reuse kernel, fp32: resident weights, R = 8 / 4 / 2 / 1, stacked taps on and off
    _case("v2_r8_stack", 32, 32, dict(V2F, mode=0, resident=1, R=8, stack=1, epi_wg=2, out_bufs=1)),
    _case("v2_r8_nostack", 32, 32, dict(mode=0, resident=1, R=8, stack=0), env={"SCI_CONV_STACK": "0"}),
    _case("v2_r4_stack", 64, 64, dict(mode=0, resident=1, R=4, stack=1, epi_wg=1, out_bufs=1)),
    _case("v2_r4_nostack", 32, 64, dict(mode=0, resident=1, R=4, stack=0), env={"SCI_CONV_STACK": "0"}),
    _case("v2_r2_stack", 32, 64, dict(mode=0, resident=1, R=2, stack=1), env={"SCI_CONV_ROWS": "2"}, round_tf32=1),
    _case("v2_r1", 32, 32, dict(mode=0, resident=1, R=1, stack=0), env={"SCI_CONV_ROWS": "1"}),
    # streamed weights: R = 1, and the two-row pairing that needs >= 8 x 148 two-row tiles
    _case("v2_streamed_r1", 96, 96, dict(mode=0, resident=0, R=1, stack=0, epi_wg=1, out_bufs=2)),
    _case("v2_resident0_r1", 32, 32, dict(mode=0, resident=0, R=1), env={"SCI_CONV_RESIDENT": "0"}),
    _case("v2_streamed_r2", 128, 128, dict(mode=0, resident=0, R=2, epi_wg=1), H=601, round_tf32=1),
    # epilogue warpgroups, TF32-rounded stores, skip-add (MODE 1), 256 columns as two passes
    _case("v2_epi1", 32, 32, dict(mode=0, epi_wg=1, out_bufs=2, resident=1), env={"SCI_CONV_EPI_WG": "1"}),
    _case("v2_epi2", 64, 64, dict(mode=0, epi_wg=2, out_bufs=1), env={"SCI_CONV_EPI_WG": "2"}),
    _case("v2_r4_round", 64, 64, dict(mode=0, resident=1, R=4), round_tf32=1),
    _case("v2_mode1_res_epi2", 32, 32, dict(mode=1, epi_wg=2), res=True),
    _case("v2_mode1_res", 32, 64, dict(mode=1, epi_wg=2), res=True, round_tf32=1),
    _case("v2_256_ps_res", 128, 256, dict(mode=1, ps=1), ps=1, relu=0, affine=False, res=True, n_plans=2),
    _case("v2_256_res", 64, 256, dict(mode=1, ps=0), res=True, n_plans=2),
    # generation-1 tile kernel
    _case("v1_s2_odd", 32, 64, dict(stride=2, half=0), kernel="v1", stride=2, H=37, W=301, round_tf32=1),
    _case("v1_cout16", 32, 16, dict(stride=1, half=0), kernel="v1"),
    _case("v1_forced_ps_res", 64, 128, dict(ps=1), kernel="v1", env={"SCI_CONV_V2": "0"}, ps=1, relu=0, res=True),
    _case("v1_forced_mode_res", 64, 64, dict(ps=0), kernel="v1", env={"SCI_CONV_V2": "0"}, res=True),
    # (split forms store fp32, or value + remainder: a TF32-rounded output would hide the products they add)
    _case("v1_wsplit", 32, 64, dict(wsplit=1, lo_chunk0=0), kernel="v1", form="wsplit"),
    _case("v1_lo_acc1", 64, 64, dict(wsplit=1, lo_chunk0=1, emit_lo=1), kernel="v1", form="lo", round_tf32=1, emit_lo=1),
    _case("v1_lo_acc0", 64, 64, dict(wsplit=1, lo_chunk0=0), kernel="v1", form="lo", env={"SCI_CONV_SPLIT_ACC": "0"}),
    _case("v1_emit_lo", 64, 64, dict(emit_lo=1), kernel="v1", round_tf32=1, emit_lo=1),
    _case("v1_f16_s2_tps3", 64, 64, dict(half=1, stride=2, tps=3), kernel="v1", form="f16", stride=2, H=37, W=301),
    _case("v1_f16_s2_tps1", 64, 64, dict(half=1, stride=2, tps=1), kernel="v1", form="f16", stride=2, H=37, W=301,
          env={"SCI_CONV_TPS": "1"}),
    # fp16 row-reuse kernel
    _case("f16_rb128", 64, 64, dict(half=1, mode=0, rb="128/128"), form="f16"),
    _case("f16_rb64", 32, 32, dict(half=1, mode=0, rb="64/64"), form="f16"),
    _case("f16_cin_store96", 128, 64, dict(half=1, rb="128/128", ks_last=2), form="f16", cin_store=96, k_used=90),
    _case("f16_cin_store96_fill", 128, 64, dict(half=1, rb="128/128", ks_last=4), form="f16", cin_store=96, fill=True),
    _case("f16_cout_store64", 64, 32, dict(half=1, rb="128/128"), form="f16", cout_store=64),
    _case("f16_cout96", 64, 96, dict(half=1), form="f16", cout_store=96),
    _case("f16_ps32_res", 64, 128, dict(half=1, ps=1, mode=1, rb="128/64"), form="f16", ps=1, relu=0, affine=False,
          res=True),
    _case("f16_ps64_res", 128, 256, dict(half=1, ps=1, mode=1, rb="128/128"), form="f16", ps=1, relu=0, affine=False,
          res=True, n_plans=2),
    _case("f16_res", 64, 64, dict(half=1, mode=1), form="f16", res=True),
    _case("f16_split1", 64, 64, dict(half=1, split=1), form="hsplit", k_used=15),
    _case("f16_split2", 128, 64, dict(half=1, split=2), form="hsplit"),
    # MODE 2: planar DenBlock output
    _case("planar_f32", 64, 32, dict(half=0, mode=2), relu=0, planar=True),
    _case("planar_f16", 64, 32, dict(half=1, mode=2), form="f16", relu=0, planar=True),
    # MODE 4: data gradient with the producing layer's activation backward fused
    _case("m4_relu_s1", 64, 64, dict(mode=4), relu=0, affine=False, round_tf32=1, mask=dict(relu=1, s2=False)),
    _case("m4_relu_s12_res", 64, 64, dict(mode=4), relu=0, affine=False, round_tf32=1, res=True, mask=dict(relu=1, s2=True)),
    _case("m4_norelu_s12", 32, 32, dict(mode=4), relu=0, affine=False, round_tf32=1, mask=dict(relu=0, s2=True)),
    _case("m4_s2t_ps128", 64, 128, dict(mode=4, ps=1), relu=0, affine=False, ps=1, round_tf32=1, res=True,
          mask=dict(relu=1, s2=True), H=19, W=151),
    _case("m4_s2t_ps256", 128, 256, dict(mode=4, ps=1), relu=0, affine=False, ps=1, round_tf32=1,
          mask=dict(relu=1, s2=False), H=19, W=151, n_plans=2),
]


def _make_operands(c, g, dev):
    """Stored tensors the kernel reads and the float64 reference operands (xr, wr).  Split forms also return their parts
    (value and remainder of the activations and of the weights) and their accumulator chains (products summed, which
    products).  Returns a dict."""
    N, H, W, Cin, Cout, form = c["N"], c["H"], c["W"], c["Cin"], c["Cout"], c["form"]
    ku = c["k_used"] or (c["cin_store"] or Cin)
    o = {}

    def randn(*s):
        return torch.randn(*s, generator=g).to(dev)
    def f16(t):
        return t.half().float()
    single_chain = c["env"].get("SCI_CONV_SPLIT_ACC") == "0"
    if form == "tf32":
        x = randn(N, H, W, Cin)
        x[..., ku:] = 0
        x = tf32(x)
        w = randn(9, Cout, Cin) / math.sqrt(9 * ku)
        w[..., ku:] = 0
        w = tf32(w)
        o.update(x=x, w=w, xr=x, wr=w, K=9 * ku)
    elif form == "wsplit":
        # x is a plain TF32 operand; the weights travel as tf32(w) in taps 0..8 and tf32(w - tf32(w)) in taps 9..17, all
        # 18 x Cin products in ONE accumulator
        x = tf32(coherent((N, H, W, Cin), 1.0, tf32, g, dev))
        w = coherent((9, Cout, Cin), 1.0 / (9 * Cin), tf32, g, dev)
        wh = tf32(w)
        wl = tf32(w - wh)
        o.update(x=x, w=torch.cat([wh, wl]), xr=x, wr=w, parts=(x, None, wh, wl), chains=((18 * Cin, "all"),))
    elif form == "lo":
        # "3xTF32": the input was written with emit_lo as [tf32(v) | tf32(v - tf32(v))], the weights are packed with
        # ci_dup = C and w_split, so the kernel forms all four products.  lo_channel0 = C puts everything except
        # value x value into a second accumulator (SCI_CONV_SPLIT_ACC=0: one accumulator for all 18 x 2C products)
        C = Cin // 2
        v = coherent((N, H, W, C), 1.0, tf32, g, dev)
        w = coherent((9, Cout, C), 1.0 / (9 * C), tf32, g, dev)
        vh, wh = tf32(v), tf32(w)
        vl, wl = tf32(v - vh), tf32(w - wh)
        wd = torch.cat([w, w], 2)
        whd = tf32(wd)
        o.update(x=torch.cat([vh, vl], 3).contiguous(), w=torch.cat([whd, tf32(wd - whd)]), xr=v, wr=w, lo_channel0=C,
                 parts=(vh, vl, wh, wl),
                 chains=((18 * Cin, "all"),) if single_chain else ((9 * C, "hh"), (27 * C, "small")))
    elif form == "f16":
        cs = c["cin_store"] or Cin
        x = randn(N, H, W, cs)
        x[..., ku:] = 0
        x = x.half()
        w = randn(9, Cout, Cin) / math.sqrt(9 * Cin)
        kw = Cin if c["fill"] else ku                  # fill: weights beyond the stored channels meet TMA's zero fill
        w[..., kw:] = 0
        w = w.half()
        xr = torch.zeros(N, H, W, Cin, device=dev, dtype=torch.float64)
        xr[..., :cs] = x.double()
        o.update(x=x, w=w, xr=xr, wr=w, K=9 * kw, cin_store=cs)
    elif form == "hsplit":
        # fp16 value + remainder x 2^11 per 32-channel group: value x value in the main accumulator (16 or 32 value
        # channels per group: split = 1 or 2), value x remainder + remainder x value in the second one
        G = Cin // 64
        ku = c["k_used"] or 32 * G
        v = coherent((N, H, W, 32 * G), 1.0, f16, g, dev)
        v[..., ku:] = 0
        w = coherent((9, Cout, 32 * G), 1.0 / (9 * ku), f16, g, dev)
        w[..., ku:] = 0
        xv, xrm = half_split(v)
        wv, wrm = half_split(w)

        def interleave(a, b):                         # per group of 32 channels: [32 values | 32 remainders]
            s = a.shape[:-1]
            return torch.stack([a.view(*s, G, 32), b.view(*s, G, 32)], -2).reshape(*s, 64 * G).contiguous()
        kv = 16 if (ku <= 16 and G == 1) else 32 * G
        o.update(x=interleave(xv, xrm), w=interleave(wv, wrm), xr=v, wr=w, cin_store=64 * G,
                 parts=(xv.float(), xrm.float() / 2048, wv.float(), wrm.float() / 2048), chains=((9 * kv, "hh"), (18 * kv, "small")))
    return o


def _split_bound(o, S, stride):
    """Accumulation bound of a split form: per accumulator chain, C_ACC * (products summed) * 2^-24 * (the S of the
    products in it), plus one rounding of the epilogue's main + small addition, plus SPLIT_REL * S for the representation
    (S of the unquantised operands).  The small products are ~2^-11 of their terms, so a chain of their own (split
    accumulators) costs almost nothing; in one chain with the main products they add their count to K."""
    xh, xl, wh, wl = (None if t is None else t.double() for t in o["parts"])
    pairs = [(xh, wh), (xh, wl), (xl, wh), (xl, wl)]
    Sp = [_ref_conv(a.abs(), b.abs(), stride) if a is not None and b is not None else None for a, b in pairs]
    Sp = [t for t in Sp if t is not None]
    S_all = sum(Sp)
    eb = SPLIT_REL * S + 2.0 ** -23 * S_all
    for k, which in o["chains"]:
        eb = eb + C_ACC * k * 2.0 ** -24 * (S_all if which == "all" else (Sp[0] if which == "hh" else S_all - Sp[0]))
    return eb


def _out_layout(c):
    """(stored dtype, stored channels, GEMM channels per stored pixel Cq, output H, W)."""
    Ho, Wo = (c["H"] - 1) // c["stride"] + 1, (c["W"] - 1) // c["stride"] + 1
    Cq = c["Cout"] // 4 if c["ps"] else c["Cout"]
    oh, ow = (2 * Ho, 2 * Wo) if c["ps"] else (Ho, Wo)
    half = c["form"] in ("f16", "hsplit")
    if c["form"] == "hsplit":
        cst = 2 * c["Cout"]
    elif half:
        cst = c["cout_store"] or Cq
    else:
        cst = Cq * (2 if c["emit_lo"] else 1)
    return (torch.float16 if half else torch.float32), cst, Cq, Ho, Wo, oh, ow


def _decode(c, y):
    """Stored output -> float64 values of the Cq real channels (split forms: value + remainder)."""
    Cq = _out_layout(c)[2]
    if c["form"] == "hsplit":
        G = c["Cout"] // 32
        s = y.shape[:-1]
        yy = y.double().view(*s, G, 2, 32)
        return (yy[..., 0, :] + yy[..., 1, :] / 2048.0).reshape(*s, 32 * G)
    if c["emit_lo"]:
        return y[..., :Cq].double() + y[..., Cq:].double()
    return y[..., :Cq].double()


def _epilogue(c, gm, sc, sh, res, in1, mask):
    """float64 epilogue of GEMM results gm [N,Ho,Wo,Cout] -> (stored-layout values, planar values or None)."""
    a = gm * sc + sh
    if c["relu"]:
        a = a.clamp_min(0)
    if c["planar"]:
        return None, in1 - a[..., :3].permute(0, 3, 1, 2)
    y = _pix_shuffle(a, c["ps"])
    if res is not None:
        y = y + res
    if mask is not None and c["mask"]["relu"]:
        y = torch.where(mask > 0, y, torch.zeros_like(y))
    return y, None


def _run_fwd_case(c, capfd, monkeypatch, dev):
    g = torch.Generator().manual_seed(zlib.crc32(repr(sorted((k, str(v)) for k, v in c.items())).encode()))
    for k, v in c["env"].items():
        monkeypatch.setenv(k, v)
    o = _make_operands(c, g, dev)
    N, H, W, Cout = c["N"], c["H"], c["W"], c["Cout"]
    dt, cst, Cq, Ho, Wo, oh, ow = _out_layout(c)
    scale = (0.5 + torch.rand(Cout, generator=g)).to(dev) if c["affine"] else None
    shift = (0.1 * torch.randn(Cout, generator=g)).to(dev) if c["affine"] else None
    # padded GEMM columns (zero weights, zero shift) must come out as exact zeros
    pad_cols = []
    if not c["res"] and c["form"] != "hsplit" and not c["planar"]:
        pad_cols = [q * Cq + Cq - 1 for q in range(4)] if c["ps"] else [Cout - 1]
        for col in pad_cols:
            o["w"][:, col] = 0
            o["wr"] = o["wr"].clone()
            o["wr"][:, col] = 0
            if "parts" in o:
                o["parts"] = o["parts"][:2] + tuple(t.clone() for t in o["parts"][2:])
                for t in o["parts"][2:]:
                    t[:, col] = 0
            if shift is not None:
                shift[col] = 0
    res = None
    if c["res"]:
        res = torch.randn(N, oh, ow, cst, generator=g).to(dev)
        res = res.half() if dt == torch.float16 else res
    mask = s1 = s2 = None
    if c["mask"]:
        mask = torch.randn(N, oh, ow, cst, generator=g).to(dev)
        mask[torch.rand(mask.shape, generator=g).to(dev) < 0.25] = 0.0            # exact zeros, negatives and positives
        s1 = torch.full((Cq,), 0.25, device=dev)                                  # accumulated onto a nonzero start
        s2 = torch.full((Cq,), -0.5, device=dev) if c["mask"]["s2"] else None
    in1 = torch.randn(N, 3, H, W, generator=g).to(dev) if c["planar"] else None

    def launch(y, pl, s1_, s2_):
        d = _desc(x=o["x"], w=o["w"], scale=scale, shift=shift, residual=res, y=y, N=N, H=H, W=W, Cin=c["Cin"], Cout=Cout,
                  stride=c["stride"], relu=c["relu"], pixel_shuffle=c["ps"], round_tf32=c["round_tf32"],
                  w_split=int(c["form"] in ("wsplit", "lo", "hsplit")), emit_lo=c["emit_lo"], half_io=int(dt == torch.float16),
                  Cin_store=o.get("cin_store", 0) if dt == torch.float16 else 0,
                  Cout_store=cst if dt == torch.float16 else 0, K_used=c["k_used"], lo_channel0=o.get("lo_channel0", 0),
                  planar_in1=in1, planar_out=pl, mask_y=mask, col_s1=s1_, col_s2=s2_,
                  mask_relu=c["mask"]["relu"] if c["mask"] else 0)
        _lib().check(_launch(d), "sci_conv3x3_fwd")

    capfd.readouterr()
    outs = []
    for rep in range(2):                                   # twice: bit-identical results
        ybuf, y = _guarded((N, oh, ow, cst), dt, dev)
        pbuf = pl = None
        if c["planar"]:
            pbuf, pl = _guarded((N, 3, H, W), torch.float32, dev)
        s1_, s2_ = (s1.clone() if s1 is not None else None), (s2.clone() if s2 is not None else None)
        launch(None if c["planar"] else y, pl, s1_, s2_)
        outs.append((ybuf, y, pbuf, pl, s1_, s2_))
        if rep == 0:
            torch.cuda.synchronize()
            _assert_plan(_plans(capfd, "conv %s plan:" % c["kernel"]), c["plan"], c["n_plans"])
    torch.cuda.synchronize()
    ybuf, y, pbuf, pl, s1_, s2_ = outs[0]
    # hygiene: margins untouched, every valid element written and finite, determinism
    assert _margins_intact(ybuf if pbuf is None else pbuf), "write outside the output tensor"
    if c["planar"]:
        assert torch.isnan(y).all() and _margins_intact(ybuf)
        assert bool(torch.isfinite(pl).all())
        assert torch.equal(_bits(pl), _bits(outs[1][3]))
    else:
        assert bool(torch.isfinite(y).all()), "output elements left unwritten (NaN) or non-finite"
        assert torch.equal(_bits(y), _bits(outs[1][1])), "two runs differ"
        if dt == torch.float16 and cst > Cq and c["form"] != "hsplit":
            assert bool((y[..., Cq:] == 0).all()), "fp16 channels beyond the real columns must be exact zeros"
        if c["round_tf32"] or c["emit_lo"]:
            assert bool(((_bits(y) & 0x1FFF) == 0).all()), "TF32-rounded outputs must have 13 zero low mantissa bits"
    # float64 reference, bound
    xr, wr = o["xr"].double(), o["wr"].double()
    gm = _ref_conv(xr, wr, c["stride"])
    S = _ref_conv(xr.abs(), wr.abs(), c["stride"])
    split = "parts" in o
    eacc = _split_bound(o, S, c["stride"]) if split else C_ACC * o["K"] * 2.0 ** -24 * S
    sc = scale.double() if scale is not None else torch.ones(Cout, dtype=torch.float64, device=dev)
    sh = shift.double() if shift is not None else torch.zeros(Cout, dtype=torch.float64, device=dev)
    res64 = res.double() if res is not None else None
    in164 = in1.double() if in1 is not None else None
    ref, pref = _epilogue(c, gm, sc, sh, res64, in164, mask)
    eb_g = sc.abs() * eacc + 2.0 ** -23 * ((sc * gm).abs() + sh.abs())        # scale * acc + shift: at most two roundings
    if c["planar"]:
        eb = eb_g[..., :3].permute(0, 3, 1, 2) + 2.0 ** -24 * (in164.abs() + pref.abs())
        got, want = pl.double(), pref
    else:
        eb = _pix_shuffle(eb_g, c["ps"])
        if res64 is not None:
            eb = eb + 2.0 ** -23 * (ref.abs() + res64.abs())
        if c["form"] == "hsplit" or c["emit_lo"]:                          # value + remainder of the stored result
            eb = eb + 2.0 ** -22 * (ref.abs() + eb) + 2.0 ** -36
        elif dt == torch.float16:
            eb = eb + 2.0 ** -11 * (ref.abs() + eb) + 2.0 ** -25
        elif c["round_tf32"]:
            eb = eb + 2.0 ** -11 * (ref.abs() + eb)
        if mask is not None and c["mask"]["relu"]:
            eb = torch.where(mask > 0, eb, torch.zeros_like(eb))
        got, want = _decode(c, y), ref
    err = (got - want).abs()
    tag = "conv %s" % c["kernel"]
    mx = _report(tag, err, eb.clamp_min(1e-300))
    assert bool((err <= eb).all()), "%s: %d elements outside the bound, max(err/bound) %.3g" % (tag, int((err > eb).sum()), mx)
    if mask is not None and c["mask"]["relu"]:
        assert bool((got[mask <= 0] == 0).all()), "masked elements must be exact zeros"
    if pad_cols:
        for col in pad_cols:
            ch = col % Cq
            assert bool((got[..., ch] == 0).all()), "padded column %d must be exactly zero" % col
    # teeth 1: one 8-channel K slice of the centre tap missing at the last pixel of the last (ragged) tile
    gp = gm.clone()
    n, ho, wo, s = N - 1, Ho - 1, Wo - 1, c["stride"]
    gp[n, ho, wo] -= wr[4, :, :8] @ xr[n, ho * s, wo * s, :8]
    rp, pp = _epilogue(c, gp, sc, sh, res64, in164, mask)
    assert bool(((pp if c["planar"] else rp) - want).abs().gt(eb).any()), "bound cannot see a missing K slice"
    # teeth 2: split forms with each cross product left out on its own, and with both (the plain-precision product)
    if split:
        xh, xl, wh, wl = (None if t is None else t.double() for t in o["parts"])
        drops = {"value x weight remainder": _ref_conv(xh, wl, c["stride"])}
        if xl is not None:
            drops["activation remainder x value"] = _ref_conv(xl, wh, c["stride"])
            drops["both cross products"] = drops["value x weight remainder"] + drops["activation remainder x value"]
        for what, dg in drops.items():
            rp, pp = _epilogue(c, gm - dg, sc, sh, res64, in164, mask)
            r = ((pp if c["planar"] else rp) - want).abs() / eb.clamp_min(1e-300)
            print("    teeth, %s left out: min / max (deviation / bound) %.3g / %.3g" % (what, float(r.min()), float(r.max())))
            assert bool((r > 1).any()), "bound cannot see the %s product left out" % what
    # MODE 4 column sums over the valid pixels, accumulated onto their start values
    if c["mask"]:
        n_pix = N * oh * ow
        depth = 32 + (n_pix + 31) // 32 + 148 + 1          # warp column sum, CTA shared atomics, global atomics, start value
        d64 = want.reshape(-1, Cq)
        for s_got, s_start, wgt in ((s1_, 0.25, None), (s2_, -0.5, mask.double().reshape(-1, Cq))):
            if s_got is None:
                continue
            terms = d64 if wgt is None else d64 * wgt
            e_terms = eb.reshape(-1, Cq) * (1 if wgt is None else wgt.abs())
            want_s = s_start + terms.sum(0)
            b = e_terms.sum(0) + C_ACC * depth * 2.0 ** -24 * (terms.abs().sum(0) + abs(s_start))
            e = (s_got.double() - want_s).abs()
            _report("column sums", e, b)
            assert bool((e <= b).all()), "column sums: max err %g" % float(e.max())
            # the sums of exactly the values the kernel stored: only their own accumulation (and, for col_s2, the rounding
            # of each product dz * mask_y) separates them - tight enough to see the last ragged 32-pixel chunk left out
            yv = got if wgt is None else got * mask.double()
            own = yv.reshape(-1, Cq)
            b_own = C_ACC * depth * 2.0 ** -24 * (own.abs().sum(0) + abs(s_start)) + (0 if wgt is None else 2.0 ** -24 * own.abs().sum(0))
            e_own = (s_got.double() - (s_start + own.sum(0))).abs()
            _report("column sums vs stored", e_own, b_own)
            assert bool((e_own <= b_own).all()), "column sums differ from the sums of the stored values"
            r = (ow - 1) % 32 + 1
            chunk = yv[N - 1, oh - 1, ow - r:].sum(0).abs()
            assert bool((chunk > b_own).any()), "column-sum bound cannot see the last %d-pixel chunk left out" % r


@pytest.mark.parametrize("c", FWD_CASES)
def test_conv_plan(cuda, capfd, monkeypatch, c):
    _run_fwd_case(c, capfd, monkeypatch, cuda)


# ---- K_used: skipped MMAs only ever added exact zeros ----------------------------------------------------------------
@pytest.mark.parametrize("form,kernel,Cin,ku,stride,ks_last", [
    ("tf32", "v2", 64, 40, 1, 1), ("tf32", "v1", 64, 40, 2, 1), ("f16", "v2", 128, 72, 1, 1), ("f16", "v1", 64, 28, 2, 2)])
def test_k_used_bit_identical(cuda, capfd, form, kernel, Cin, ku, stride, ks_last):
    g = torch.Generator().manual_seed(Cin + ku)
    N, H, W, Cout = N_, H_, 301, 64
    half = form == "f16"
    x = torch.randn(N, H, W, Cin, generator=g)
    x[..., ku:] = 0
    w = torch.randn(9, Cout, Cin, generator=g) / math.sqrt(9 * ku)
    w[..., ku:] = 0
    x, w = (x.half(), w.half()) if half else (tf32(x), tf32(w))
    x, w = x.to(cuda), w.to(cuda)
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    ys = []
    for k in (0, ku):
        y = torch.full((N, Ho, Wo, Cout), float("nan"), dtype=x.dtype, device=cuda)
        d = _desc(x=x, w=w, y=y, N=N, H=H, W=W, Cin=Cin, Cout=Cout, stride=stride, relu=1, half_io=int(half), K_used=k)
        capfd.readouterr()
        _lib().check(_launch(d), "sci_conv3x3_fwd")
        torch.cuda.synchronize()
        _assert_plan(_plans(capfd, "conv %s plan:" % kernel), {"ks_last": ks_last if k else 4})
        ys.append(y)
    assert bool(torch.isfinite(ys[0]).all())
    assert torch.equal(_bits(ys[0]), _bits(ys[1]))


# ---- PDL: a dependent launch reads its predecessor's output ----------------------------------------------------------
@pytest.mark.parametrize("half", [0, 1])
def test_pdl_chain_bit_identical(cuda, capfd, half):
    g = torch.Generator().manual_seed(7 + half)
    N, H, W, C = N_, H_, W_, 64
    cast = (lambda t: t.half()) if half else tf32
    x = cast(torch.randn(N, H, W, C, generator=g)).to(cuda)
    w1 = cast(torch.randn(9, C, C, generator=g) / 24).to(cuda)
    w2 = cast(torch.randn(9, C, C, generator=g) / 24).to(cuda)
    shift = (0.1 * torch.randn(C, generator=g)).to(cuda)
    dt = x.dtype
    outs = []
    for pdl in (0, 1):
        y1 = torch.full((N, H, W, C), float("nan"), dtype=dt, device=cuda)
        Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
        # the second layer: the row-reuse kernel (fp32) or the stride-2 tile kernel (fp16)
        y2 = torch.full((N, Ho, Wo, C) if half else (N, H, W, C), float("nan"), dtype=dt, device=cuda)
        d1 = _desc(x=x, w=w1, shift=shift, y=y1, N=N, H=H, W=W, Cin=C, Cout=C, stride=1, relu=1, round_tf32=1 - half,
                   half_io=half, pdl=pdl)
        d2 = _desc(x=y1, w=w2, shift=shift, y=y2, N=N, H=H, W=W, Cin=C, Cout=C, stride=2 if half else 1, relu=1,
                   half_io=half, pdl=pdl)
        capfd.readouterr()
        _lib().check(_launch(d1), "layer 1")
        _lib().check(_launch(d2), "layer 2")
        torch.cuda.synchronize()
        err = capfd.readouterr().err
        assert ("pdl %d" % pdl) in err.splitlines()[-1], err
        outs.append((y1, y2))
    for a, b in zip(*outs):
        assert bool(torch.isfinite(a).all()) and torch.equal(_bits(a), _bits(b))


# ---- refusals: knobs and options the planner does not accept -------------------------------------------------------
def test_unsupported_combinations_refused(cuda):
    x = torch.zeros(1, 8, 8, 64, device=cuda, dtype=torch.float16)
    w = torch.zeros(9, 64, 64, device=cuda, dtype=torch.float16)
    y = torch.zeros(1, 8, 8, 128, device=cuda, dtype=torch.float16)
    m = torch.zeros(1, 8, 8, 64, device=cuda)
    base = dict(x=x, w=w, y=y, N=1, H=8, W=8, Cin=64, Cout=64, stride=1, half_io=1)
    # fused activation backward exists on the fp32 TMA-store path only
    assert _launch(_desc(**base, mask_y=m, col_s1=m)) == SCI_EUNSUPPORTED
    # fp16 split form: plain layers only
    assert _launch(_desc(**base, w_split=1, Cout_store=128, residual=y)) == SCI_EUNSUPPORTED
    # emit_lo needs round_tf32
    xf, wf, yf = torch.zeros(1, 8, 8, 64, device=cuda), torch.zeros(18, 64, 64, device=cuda), torch.zeros(1, 8, 8, 128, device=cuda)
    assert _launch(_desc(x=xf, w=wf, y=yf, N=1, H=8, W=8, Cin=64, Cout=64, stride=1, w_split=1, emit_lo=1)) == SCI_EUNSUPPORTED


# ---- FFMA reference kernel (SCI_CONV_REF): the checker of the full-size tests ---------------------------------------
@pytest.mark.parametrize("Cin,Cout,stride,ps,res", [(32, 64, 1, 0, True), (64, 32, 2, 0, False), (64, 128, 1, 1, False)])
def test_ffma_reference_kernel(cuda, Cin, Cout, stride, ps, res):
    g = torch.Generator().manual_seed(Cin * Cout + stride)
    N, H, W = N_, H_, 301
    x = torch.randn(N, H, W, Cin, generator=g).to(cuda)
    w = (torch.randn(9, Cout, Cin, generator=g) / math.sqrt(9 * Cin)).to(cuda)
    sc, sh = (0.5 + torch.rand(Cout, generator=g)).to(cuda), (0.1 * torch.randn(Cout, generator=g)).to(cuda)
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    oh, ow, Cq = (2 * Ho, 2 * Wo, Cout // 4) if ps else (Ho, Wo, Cout)
    r = torch.randn(N, oh, ow, Cq, generator=g).to(cuda) if res else None
    buf, y = _guarded((N, oh, ow, Cq), torch.float32, cuda)
    d = _desc(x=x, w=w, scale=sc, shift=sh, residual=r, y=y, N=N, H=H, W=W, Cin=Cin, Cout=Cout, stride=stride, relu=1,
              pixel_shuffle=ps)
    _lib().check(_launch(d, impl=1), "sci_conv3x3_fwd(ref)")
    torch.cuda.synchronize()
    assert _margins_intact(buf) and bool(torch.isfinite(y).all())
    gm = _ref_conv(x.double(), w.double(), stride)
    S = _ref_conv(x.double().abs(), w.double().abs(), stride)
    a = (gm * sc.double() + sh.double()).clamp_min(0)
    ref = _pix_shuffle(a, ps) + (r.double() if res else 0)
    # at most one rounding per product and one per accumulation step (fused or not): (K + 1) * 2^-24 * S <= C_ACC * K * ...
    eb = _pix_shuffle(sc.double() * C_ACC * 9 * Cin * 2.0 ** -24 * S + 2.0 ** -23 * ((sc.double() * gm).abs() + sh.double().abs()), ps)
    if res:
        eb = eb + 2.0 ** -23 * (ref.abs() + r.double().abs())
    err = (y.double() - ref).abs()
    _report("conv ref", err, eb)
    assert bool((err <= eb).all())
    gp = gm.clone()
    gp[N - 1, Ho - 1, Wo - 1] -= w.double()[4, :, :8] @ x.double()[N - 1, (Ho - 1) * stride, (Wo - 1) * stride, :8]
    rp = _pix_shuffle((gp * sc.double() + sh.double()).clamp_min(0), ps) + (r.double() if res else 0)
    assert bool(((rp - ref).abs() > eb).any())


# ---- weight gradient ------------------------------------------------------------------------------------------------
WGRAD_CASES = [
    # id, Cin, Cout, stride, N, H, W, env, plan prefix, expected plan fields
    ("v3_cp32", 32, 64, 1, N_, H_, W_, {}, "wgrad v3", dict(cp=32, cq=64, p_is_dz=0)),
    ("v3_cp64", 64, 64, 1, N_, H_, W_, {}, "wgrad v3", dict(cp=64, cq=64, p_is_dz=1)),
    ("v3_cq96", 96, 32, 1, N_, H_, W_, {}, "wgrad v3", dict(cp=32, cq=96, p_is_dz=1)),
    ("v3_many_tiles", 32, 32, 1, N_, 250, 301, {}, "wgrad v3", dict(cp=32, cq=32)),
    ("v2_swap_fuse", 32, 32, 1, N_, H_, W_, {"SCI_WGRAD_V3": "0"}, "wgrad v2", dict(swap=1, fuse=1, m_tiles=1)),
    ("v2_swap", 128, 64, 1, N_, H_, W_, {}, "wgrad v2", dict(swap=1, fuse=0, accs=3)),
    ("v2_fuse", 64, 128, 1, N_, H_, W_, {}, "wgrad v2", dict(swap=0, fuse=1, m_tiles=1)),
    ("v2_nofuse", 128, 128, 1, N_, H_, W_, {}, "wgrad v2", dict(swap=0, fuse=0, m_tiles=1, accs=3)),
    ("v2_two_m_tiles", 128, 256, 1, N_, H_, W_, {}, "wgrad v2", dict(swap=0, m_tiles=2)),
    ("v2_stride2", 64, 128, 2, N_, 37, 301, {}, "wgrad v2", dict(swap=0, fuse=1, stride=2)),
    ("v2_many_tiles", 64, 128, 1, N_, 250, 301, {}, "wgrad v2", dict(swap=0, fuse=1)),
    ("v2_fuse_v3_off", 64, 64, 1, N_, H_, W_, {"SCI_WGRAD_V3": "0"}, "wgrad v2", dict(swap=0, fuse=1, m_tiles=1)),
    ("v2_stride2_two_m", 32, 256, 2, N_, 37, 301, {}, "wgrad v2", dict(swap=0, fuse=1, m_tiles=2, stride=2)),
]


@pytest.mark.parametrize("c", [pytest.param(c, id=c[0]) for c in WGRAD_CASES])
def test_wgrad_plan(cuda, capfd, monkeypatch, c):
    from adaptivepnp_sci_b200 import engine
    cid, Cin, Cout, stride, N, H, W, env, prefix, want = c
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    g = torch.Generator().manual_seed(Cin * 7 + Cout + stride)
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    x = tf32(torch.randn(N, H, W, Cin, generator=g)).to(cuda)
    dz = tf32(torch.randn(N, Ho, Wo, Cout, generator=g)).to(cuda)
    osc = (0.5 + torch.rand(Cout, generator=g)).to(cuda)
    dw0 = torch.randn(9, Cout, Cin, generator=g).to(cuda)                 # the gradient is ACCUMULATED onto this
    buf, dw = _guarded((9, Cout, Cin), torch.float32, cuda)
    dw.copy_(dw0)
    d = engine.WgradDesc(x.data_ptr(), dz.data_ptr(), osc.data_ptr(), dw.data_ptr(), N, H, W, Cin, Cout, stride)
    capfd.readouterr()
    _lib().check(_lib().lib.sci_conv3x3_wgrad(ctypes.byref(d), 0, _lib().stream()), "sci_conv3x3_wgrad")
    torch.cuda.synchronize()
    plans = _plans(capfd, prefix + " plan:")
    _assert_plan(plans, want)
    assert _margins_intact(buf) and bool(torch.isfinite(dw).all())
    # float64: dw[3r+s][co][ci] = dw0 + osc[co] * sum_p dz[p][co] * x[p*stride + (r-1, s-1)][ci]
    xp = F.pad(x.double(), (0, 0, 1, 1, 1, 1))
    dz64 = dz.double().reshape(-1, Cout)
    sums, S = [], []
    for r in range(3):
        for s in range(3):
            xs = xp[:, r:r + stride * (Ho - 1) + 1:stride, s:s + stride * (Wo - 1) + 1:stride].reshape(-1, Cin)
            sums.append(dz64.t() @ xs)
            S.append(dz64.abs().t() @ xs.abs())
    gsum, S = torch.stack(sums), torch.stack(S)
    o64 = osc.double()[None, :, None]
    ref = dw0.double() + o64 * gsum
    # a term's path: the MMA that forms it (<= 8 products of one K step), the TMEM accumulator of its CTA (8 MMAs per 8x8
    # tile over the tiles the CTA owns), the CTAs' reductions into dw, and the initial value: C_ACC * depth * 2^-24 * S
    p = plans[0]
    depth = 8 + 8 * -(-p["tiles"] // p["grid"]) + p["grid"] + 1
    eb = o64 * C_ACC * depth * 2.0 ** -24 * S + 2.0 ** -23 * ((o64 * gsum).abs() + ref.abs())
    err = (dw.double() - ref).abs()
    _report(cid, err, eb)
    assert bool((err <= eb).all()), "max err/bound %g" % float((err / eb).max())
    # teeth: the last (ragged) 8x8 tile of the last image missing from every sum
    h0, w0 = (Ho - 1) // 8 * 8, (Wo - 1) // 8 * 8
    dzt = dz.double()[N - 1, h0:, w0:].reshape(-1, Cout)
    drop = []
    for r in range(3):
        for s in range(3):
            xs = xp[N - 1, r + stride * h0:r + stride * (Ho - 1) + 1:stride, s + stride * w0:s + stride * (Wo - 1) + 1:stride]
            drop.append(dzt.t() @ xs.reshape(-1, Cin))
    assert bool(((o64 * torch.stack(drop)).abs() > eb).any()), "bound cannot see one missing tile"


# ---- packers: numpy restatements, bit for bit ------------------------------------------------------------------------
def np_tf32(v):
    b = np.asarray(v, np.float32).view(np.uint32)
    return ((b + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)


def np_pack(w, Co, Ci, groups, Co_pad, Ci_pad, ps, oscale, tflip, round_tf32, ci_dup):
    total = 9 * Co_pad * Ci_pad
    idx = np.arange(total)
    if not tflip:
        ci, col, tap = idx % Ci_pad, (idx // Ci_pad) % Co_pad, idx // (Ci_pad * Co_pad)
    else:
        col, ci, tap = idx % Co_pad, (idx // Co_pad) % Ci_pad, idx // (Ci_pad * Co_pad)
    if ci_dup > 0:
        ci = np.where((ci >= ci_dup) & (ci < ci_dup + Ci), ci - ci_dup, ci)
    q = Co_pad >> 2
    co = (col % q) * 4 + col // q if ps else col
    ok = (((col % q) < (Co >> 2)) if ps else (col < Co)) & (ci < Ci)
    cig, cog = Ci // groups, Co // groups
    grp = co // cog
    ok &= (ci // cig) == grp
    src = 8 - tap if tflip else tap
    wi = np.where(ok, (co * cig + (ci - grp * cig)) * 9 + src, 0)
    v = np.where(ok, w.reshape(-1)[wi], np.float32(0)).astype(np.float32)
    if tflip and oscale is not None:
        v = (v * oscale[col]).astype(np.float32)
    if round_tf32 == 2:
        hi = np_tf32(v)
        return np.concatenate([hi, np_tf32((v - hi).astype(np.float32))])
    return np_tf32(v) if round_tf32 else v


def np_pack_half(w, Co, Ci, groups, Co_pad, Ci_pad, ps, ci_dup):
    total = 9 * Co_pad * Ci_pad
    idx = np.arange(total)
    ci, col, tap = idx % Ci_pad, (idx // Ci_pad) % Co_pad, idx // (Ci_pad * Co_pad)
    if ci_dup > 0:
        ci = np.where((ci >= ci_dup) & (ci < ci_dup + Ci), ci - ci_dup, ci)
    part = (ci >> 5) & 1 if ci_dup == -1 else np.zeros_like(ci)
    if ci_dup == -1:
        ci = ((ci >> 6) << 5) | (ci & 31)
    q = Co_pad >> 2
    co = (col % q) * 4 + col // q if ps else col
    ok = (((col % q) < (Co >> 2)) if ps else (col < Co)) & (ci < Ci)
    cig, cog = Ci // groups, Co // groups
    grp = co // cog
    ok &= (ci // cig) == grp
    wi = np.where(ok, (co * cig + (ci - grp * cig)) * 9 + tap, 0)
    v = np.where(ok, w.reshape(-1)[wi], np.float32(0)).astype(np.float32)
    rem = ((v - v.astype(np.float16).astype(np.float32)) * np.float32(2048)).astype(np.float32)
    return np.where(part == 1, rem, v).astype(np.float16)


def np_pack_s2t(w, Co, Ci, Co_pad, Ci_pad, oscale, round_tf32):
    total = 9 * 4 * Ci_pad * Co_pad
    idx = np.arange(total)
    co, col, tap = idx % Co_pad, (idx // Co_pad) % (4 * Ci_pad), idx // (Co_pad * 4 * Ci_pad)
    q, ci = col // Ci_pad, col % Ci_pad

    def src(par, d):
        return np.where(par == 0, np.where(d == 0, 1, -1), np.where(d == 0, 2, np.where(d == 1, 0, -1)))
    kh, kw = src(q >> 1, tap // 3 - 1), src(q & 1, tap % 3 - 1)
    ok = (co < Co) & (ci < Ci) & (kh >= 0) & (kw >= 0)
    wi = np.where(ok, (co * Ci + ci) * 9 + kh * 3 + kw, 0)
    v = np.where(ok, w.reshape(-1)[wi], np.float32(0)).astype(np.float32)
    if oscale is not None:
        v = (v * oscale[np.minimum(co, len(oscale) - 1)]).astype(np.float32)
    return np_tf32(v) if round_tf32 else v


def np_unpack(packed, Co, Ci, groups, Co_pad, Ci_pad, ps, ci_dup):
    cig, cog = Ci // groups, Co // groups
    idx = np.arange(Co * cig * 9)
    tap, cil, co = idx % 9, (idx // 9) % cig, idx // (9 * cig)
    ci = (co // cog) * cig + cil
    col = (co & 3) * (Co_pad >> 2) + (co >> 2) if ps else co
    base = (tap * Co_pad + col) * Ci_pad + ci
    gsum = packed[base]
    if ci_dup > 0:
        gsum = (gsum + packed[base + ci_dup]).astype(np.float32)
    return gsum


def _tie_weights(g, Co, cig):
    """Random weights with TF32 and fp16 rounding ties planted in them."""
    w = torch.randn(Co, cig, 3, 3, generator=g).numpy().astype(np.float32)
    ties = np.array([1 + 2 ** -11, -(1 + 2 ** -11), 1 + 3 * 2 ** -11, -(1 + 3 * 2 ** -11), 0.5 + 2 ** -12,
                     3 * 2 ** -20 + 2 ** -31, 1 + 2 ** -11 + 2 ** -23], np.float32)
    flat = w.reshape(-1)
    flat[:len(ties)] = ties
    return w


def test_rounding_restatements_at_ties():
    """The numpy roundings the packer checks rely on: TF32 RNA (ties away from zero) and fp16 round-to-nearest-even."""
    assert np_tf32(np.float32(1 + 2 ** -11)) == np.float32(1 + 2 ** -10)
    assert np_tf32(np.float32(-(1 + 2 ** -11))) == np.float32(-(1 + 2 ** -10))
    assert np_tf32(np.float32(1 + 3 * 2 ** -11)) == np.float32(1 + 2 ** -9)
    assert np_tf32(np.float32(1 + 2 ** -11 - 2 ** -23)) == np.float32(1)
    assert np.float32(1 + 2 ** -11).astype(np.float16) == np.float16(1)
    assert np.float32(1 + 3 * 2 ** -11).astype(np.float16) == np.float16(1 + 2 ** -9)
    assert np.float32(1 + 2 ** -11 + 2 ** -23).astype(np.float16) == np.float16(1 + 2 ** -10)
    # and the torch helper of the conv cases agrees with the numpy one
    v = torch.randn(4096, generator=torch.Generator().manual_seed(3))
    v[:4] = torch.tensor([1 + 2 ** -11, -(1 + 2 ** -11), 1 + 3 * 2 ** -11, 2 ** -126 + 2 ** -138])
    assert np.array_equal(tf32(v).numpy().view(np.uint32), np_tf32(v.numpy()).view(np.uint32))


PACK_CASES = [
    # Co, Ci, groups, Co_pad, Ci_pad, ps, tflip, oscale, round_tf32, ci_dup
    (96, 15, 1, 96, 32, 0, 0, False, 1, 16),          # first layer, remainder copy of the input
    (90, 12, 3, 96, 32, 0, 0, False, 1, 0),           # grouped input conv
    (256, 128, 1, 256, 128, 1, 0, False, 1, 0),       # PixelShuffle column permutation
    (12, 96, 1, 32, 96, 1, 0, False, 2, 0),           # PixelShuffle, split taps
    (64, 32, 1, 64, 32, 0, 1, True, 1, 0),            # transpose + flip + oscale
    (90, 12, 3, 96, 32, 0, 1, True, 0, 16),           # grouped, transposed, duplicated, unrounded
    (96, 96, 1, 96, 192, 0, 0, False, 2, 96),         # 3xTF32 layer: split taps, duplicated input
]


@pytest.mark.parametrize("c", PACK_CASES)
def test_pack_weights_bit_exact(cuda, c):
    from adaptivepnp_sci_b200._lib import call, ptr, stream
    Co, Ci, groups, Co_pad, Ci_pad, ps, tflip, use_os, rt, dup = c
    g = torch.Generator().manual_seed(Co * Ci + rt)
    w = _tie_weights(g, Co, Ci // groups)
    osc = (0.5 + torch.rand(Co_pad, generator=g)).numpy().astype(np.float32) if use_os else None
    out = torch.full(((18 if rt == 2 else 9) * Co_pad * Ci_pad,), float("nan"), device=cuda)
    wd = torch.from_numpy(w).to(cuda)
    od = torch.from_numpy(osc).to(cuda) if use_os else None
    call("sci_conv_pack_weights", ptr(wd), ptr(out), Co, Ci, groups, Co_pad, Ci_pad, ps, ptr(od), tflip, rt, dup, stream())
    want = np_pack(w, Co, Ci, groups, Co_pad, Ci_pad, ps, osc, tflip, rt, dup)
    assert np.array_equal(out.cpu().numpy().view(np.uint32), want.view(np.uint32))


@pytest.mark.parametrize("c", [(96, 15, 1, 96, 64, 0, -1), (96, 96, 1, 96, 192, 0, -1), (90, 12, 3, 96, 64, 0, 16),
                               (256, 128, 1, 256, 128, 1, 0), (128, 32, 1, 128, 32, 1, 0)])
def test_pack_weights_half_bit_exact(cuda, c):
    from adaptivepnp_sci_b200._lib import call, ptr, stream
    Co, Ci, groups, Co_pad, Ci_pad, ps, dup = c
    g = torch.Generator().manual_seed(Co + Ci + dup)
    w = _tie_weights(g, Co, Ci // groups)
    out = torch.empty(9 * Co_pad * Ci_pad, dtype=torch.float16, device=cuda)
    wd = torch.from_numpy(w).to(cuda)
    call("sci_conv_pack_weights_half", ptr(wd), ptr(out), Co, Ci, groups, Co_pad, Ci_pad, ps, dup, stream())
    want = np_pack_half(w, Co, Ci, groups, Co_pad, Ci_pad, ps, dup)
    assert np.array_equal(out.cpu().numpy().view(np.uint16), want.view(np.uint16))


@pytest.mark.parametrize("c", [(64, 32, 64, 32, True, 1), (128, 64, 128, 64, False, 0), (40, 20, 64, 32, True, 1)])
def test_pack_weights_s2t_bit_exact(cuda, c):
    from adaptivepnp_sci_b200._lib import call, ptr, stream
    Co, Ci, Co_pad, Ci_pad, use_os, rt = c
    g = torch.Generator().manual_seed(Co * 3 + Ci)
    w = _tie_weights(g, Co, Ci)
    osc = (0.5 + torch.rand(Co_pad, generator=g)).numpy().astype(np.float32) if use_os else None
    out = torch.empty(36 * Co_pad * Ci_pad, device=cuda)
    wd = torch.from_numpy(w).to(cuda)
    od = torch.from_numpy(osc).to(cuda) if use_os else None
    call("sci_conv_pack_weights_s2t", ptr(wd), ptr(out), Co, Ci, Co_pad, Ci_pad, ptr(od), rt, stream())
    want = np_pack_s2t(w, Co, Ci, Co_pad, Ci_pad, osc, rt)
    assert np.array_equal(out.cpu().numpy().view(np.uint32), want.view(np.uint32))


@pytest.mark.parametrize("c", [(96, 15, 1, 96, 32, 0, 16), (90, 12, 3, 96, 32, 0, 0), (256, 128, 1, 256, 128, 1, 0),
                               (12, 96, 1, 32, 192, 1, 96)])
def test_unpack_wgrad_bit_exact(cuda, c):
    from adaptivepnp_sci_b200._lib import call, ptr, stream
    Co, Ci, groups, Co_pad, Ci_pad, ps, dup = c
    g = torch.Generator().manual_seed(Co + 5 * Ci)
    packed = torch.randn(9 * Co_pad * Ci_pad, generator=g)
    out = torch.full((Co * (Ci // groups) * 9,), float("nan"), device=cuda)
    pd = packed.to(cuda)
    call("sci_conv_unpack_wgrad", ptr(pd), ptr(out), Co, Ci, groups, Co_pad, Ci_pad, ps, dup, stream())
    want = np_unpack(packed.numpy(), Co, Ci, groups, Co_pad, Ci_pad, ps, dup)
    assert np.array_equal(out.cpu().numpy().view(np.uint32), want.view(np.uint32))


def test_layer_ops_batch_equals_single_calls(cuda):
    """One table entry of every kind equals the corresponding single call bit for bit."""
    from adaptivepnp_sci_b200 import engine
    from adaptivepnp_sci_b200._lib import call, ptr, stream
    g = torch.Generator().manual_seed(11)
    Co, Ci, Co_pad, Ci_pad = 96, 40, 96, 64
    w = torch.from_numpy(_tie_weights(g, Co, Ci)).to(cuda)
    osc = (0.5 + torch.rand(Co_pad, generator=g)).to(cuda)
    pk = torch.randn(9 * Co_pad * Ci_pad, generator=g).to(cuda)
    gam, bet, mean = (torch.randn(Co, generator=g).to(cuda) for _ in range(3))
    var = torch.rand(Co, generator=g).to(cuda) + 0.1
    s1, s2 = torch.randn(Co, generator=g).to(cuda), torch.randn(Co, generator=g).to(cuda)
    n9 = 9 * Co_pad * Ci_pad

    def outs():
        return dict(p0=torch.full((n9,), float("nan"), device=cuda), p0t=torch.full((n9,), float("nan"), device=cuda),
                    p1=torch.full((4 * n9,), float("nan"), device=cuda),
                    p2=torch.full((n9,), float("nan"), device=cuda, dtype=torch.float16),
                    p3=torch.full((Co * Ci * 9,), float("nan"), device=cuda),
                    sc=torch.full((Co_pad,), float("nan"), device=cuda), sh=torch.full((Co_pad,), float("nan"), device=cuda),
                    dg=torch.full((Co,), float("nan"), device=cuda), db=torch.full((Co,), float("nan"), device=cuda),
                    cp=torch.full((Co,), float("nan"), device=cuda))
    a, b = outs(), outs()
    call("sci_conv_pack_weights", ptr(w), ptr(a["p0"]), Co, Ci, 1, Co_pad, Ci_pad, 0, None, 0, 1, 0, stream())
    call("sci_conv_pack_weights", ptr(w), ptr(a["p0t"]), Co, Ci, 1, Co_pad, Ci_pad, 0, ptr(osc), 1, 1, 0, stream())
    call("sci_conv_pack_weights_s2t", ptr(w), ptr(a["p1"]), Co, Ci, Co_pad, Ci_pad, ptr(osc), 1, stream())
    call("sci_conv_pack_weights_half", ptr(w), ptr(a["p2"]), Co, Ci, 1, Co_pad, Ci_pad, 0, 0, stream())
    call("sci_conv_unpack_wgrad", ptr(pk), ptr(a["p3"]), Co, Ci, 1, Co_pad, Ci_pad, 0, 0, stream())
    call("sci_bn_fold", ptr(gam), ptr(bet), ptr(mean), ptr(var), 1e-5, ptr(a["sc"]), ptr(a["sh"]), Co, Co_pad, stream())
    call("sci_bn_param_grad", ptr(s1), ptr(s2), ptr(gam), ptr(bet), ptr(a["dg"]), ptr(a["db"]), Co, stream())
    a["cp"].copy_(s1)
    ops = [engine._op(0, Co, Ci, 1, Co_pad, Ci_pad, 0, 0, 1, 0, a=w, o0=b["p0"]),
           engine._op(0, Co, Ci, 1, Co_pad, Ci_pad, 0, 1, 1, 0, a=w, b=osc, o0=b["p0t"]),
           engine._op(1, Co=Co, Ci=Ci, Co_pad=Co_pad, Ci_pad=Ci_pad, round_tf32=1, a=w, b=osc, o0=b["p1"]),
           engine._op(2, Co, Ci, 1, Co_pad, Ci_pad, 0, a=w, o0=b["p2"]),
           engine._op(3, Co, Ci, 1, Co_pad, Ci_pad, 0, a=pk, o0=b["p3"]),
           engine._op(4, Co=Co, Co_pad=Co_pad, eps=1e-5, a=gam, b=bet, c=mean, d=var, o0=b["sc"], o1=b["sh"]),
           engine._op(5, Co=Co, a=s1, b=s2, c=gam, d=bet, o0=b["dg"], o1=b["db"]),
           engine._op(6, Co=Co, a=s1, o0=b["cp"])]
    engine.OpTable(ops, cuda).run()
    torch.cuda.synchronize()
    for k in a:
        assert torch.equal(_bits(a[k]), _bits(b[k])), k


# ---- the networks' own layers ---------------------------------------------------------------------------------------
def _network_engines(monkeypatch):
    """(name, engine) for every network engine and inference form; the layer lists are the engines' own."""
    from adaptivepnp_sci_b200 import engine
    from adaptivepnp_sci_b200.fastdvdnet_models import FastDVDnet
    from adaptivepnp_sci_b200.ffdnet_ipol_models import FFDNet as FFDNetIPOL
    from adaptivepnp_sci_b200.network_demosaicking import DDnet
    from adaptivepnp_sci_b200.network_ffdnet import FFDNet
    torch.manual_seed(0)
    out = [("ffdnet_colour", engine.FFDNetEngine(FFDNet(3, 3, 96, 12, 'R').cuda())),
           ("ffdnet_gray", engine.FFDNetEngine(FFDNet(1, 1, 64, 15, 'R').cuda())),
           ("ffdnet_ipol", engine.FFDNetEngine(FFDNetIPOL(1).cuda().eval())),
           ("ddnet", engine.DDnetEngine(DDnet().cuda()))]
    monkeypatch.setenv("SCI_FFDNET_INF", "tf32")                  # the 3xTF32 inference chain
    out.append(("ffdnet_colour_3xtf32", engine.FFDNetEngine(FFDNet(3, 3, 96, 12, 'R').cuda())))
    monkeypatch.delenv("SCI_FFDNET_INF")
    for sw in ("1", "0"):
        monkeypatch.setenv("SCI_CONV_SW64", sw)
        out.append(("fastdvdnet_sw64_%s" % sw, engine.FastDVDnetEngine(FastDVDnet(5).cuda())))
    monkeypatch.delenv("SCI_CONV_SW64")
    return out


def _layer_check(L, dev, g, tag, capfd):
    """One forward launch of a network layer (ConvLayer or HalfLayer) at a ragged size against float64 of the operands
    the kernel multiplies (its packed weights)."""
    from adaptivepnp_sci_b200 import engine
    N, H, W = N_, 21, 262
    if isinstance(L, engine.HalfLayer):
        b = L.base
        half, K, Cout, split = True, L.K, L.N, L.split
        cs = L.cin_store
        ku = L.k_used
        v = torch.randn(N, H, W, cs if not split else cs // 2, generator=g).to(dev)
        if split:
            G = cs // 64
            v[..., b.Ci:] = 0
            xv, xr_ = half_split(v)
            x = torch.stack([xv.view(N, H, W, G, 32), xr_.view(N, H, W, G, 32)], -2).reshape(N, H, W, cs).contiguous()
            wk = L.wpk.view(9, Cout, G, 2, 32).double()
            wr = (wk[:, :, :, 0] + wk[:, :, :, 1] / 2048.0).reshape(9, Cout, 32 * G)
            xr, Kc = v.double(), 18 * K
        else:
            v[..., ku:] = 0
            x = v.half()
            xr = torch.zeros(N, H, W, K, dtype=torch.float64, device=dev)
            xr[..., :cs] = x.double()
            wr, Kc = L.wpk.view(9, Cout, K).double(), 9 * ku
        stride, relu, ps = L.stride, L.relu, L.ps
        cst = L.cout_store
        d = dict(Cin=K, half_io=1, w_split=int(split), Cin_store=cs, Cout_store=cst, K_used=ku)
    else:
        b = L
        half, K, Cout, split = False, L.Ci_pad, L.Co_pad, False
        x = tf32(torch.randn(N, H, W, K, generator=g)).to(dev)
        taps = L.wpk.numel() // (9 * Cout * K)       # 2: value + remainder weights (w_split)
        wr = L.wpk.view(taps, 9, Cout, K).double().sum(0)        # value + remainder taps: both products are exact
        xr, Kc = x.double(), 9 * taps * K
        stride, relu, ps = L.stride, L.relu, L.ps
        cst = Cout // 4 if ps else Cout
        d = dict(Cin=K, w_split=int(taps == 2), lo_channel0=L.ci_half if L.dup_in else 0)
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    oh, ow = (2 * Ho, 2 * Wo) if ps else (Ho, Wo)
    Cq = Cout // 4 if ps else Cout
    ybuf, y = _guarded((N, oh, ow, cst), torch.float16 if half else torch.float32, dev)
    desc = _desc(x=x, w=L.wpk, scale=b.scale, shift=b.shift, y=y, N=N, H=H, W=W, Cout=Cout, stride=stride, relu=int(relu),
                 pixel_shuffle=int(ps), **d)
    capfd.readouterr()
    _lib().check(_launch(desc), "sci_conv3x3_fwd " + tag)
    torch.cuda.synchronize()
    # the plan the planner must pick for this layer (fwd2_eligible): the row-reuse kernel for stride-1 layers except the
    # fp32 split-weight ones, two passes of 128 columns for Cout = 256
    if half:
        kern = "v2" if stride == 1 else "v1"
    else:
        kern = "v2" if (stride == 1 and taps == 1 and Cout % 32 == 0 and (Cout <= 128 or Cout == 256)) else "v1"
    _assert_plan(_plans(capfd, "conv %s plan:" % kern), dict(half=int(half)), 2 if kern == "v2" and Cout > 128 else 1)
    assert _margins_intact(ybuf) and bool(torch.isfinite(y).all()), tag
    sc = b.scale.double() if b.scale is not None else torch.ones(Cout, dtype=torch.float64, device=dev)
    sh = b.shift.double() if b.shift is not None else torch.zeros(Cout, dtype=torch.float64, device=dev)
    gm = _ref_conv(xr, wr, stride)
    S = _ref_conv(xr.abs(), wr.abs(), stride)
    def epi(g_):
        a = g_ * sc + sh
        return _pix_shuffle(a.clamp_min(0) if relu else a, ps)
    ref = epi(gm)
    eb = _pix_shuffle(sc.abs() * (C_ACC * Kc * 2.0 ** -24 + (SPLIT_REL if split else 0)) * S
                      + 2.0 ** -23 * ((sc * gm).abs() + sh.abs()), ps)
    if split:
        G = Cout // 32
        yy = y.double().view(N, oh, ow, G, 2, 32)
        got = (yy[..., 0, :] + yy[..., 1, :] / 2048.0).reshape(N, oh, ow, Cout)
        eb = eb + 2.0 ** -22 * (ref.abs() + eb) + 2.0 ** -36
    else:
        got = y[..., :Cq].double()
        eb = eb + (2.0 ** -11 * (ref.abs() + eb) + 2.0 ** -25 if half else 2.0 ** -24 * ref.abs())
        if half and cst > Cq:
            assert bool((y[..., Cq:] == 0).all()), tag
    err = (got - ref).abs()
    r = err / eb.clamp_min(1e-300)
    mx, rms = float(r.max()), float(torch.sqrt((r * r).mean()))
    assert bool((err <= eb).all()), "%s: max(err/bound) %.3g" % (tag, mx)
    # teeth: one 8-channel K slice of the centre tap missing at the last pixel of the last (ragged) tile
    gp = gm.clone()
    gp[N - 1, Ho - 1, Wo - 1] -= wr[4, :, :8] @ xr[N - 1, (Ho - 1) * stride, (Wo - 1) * stride, :8]
    assert bool(((epi(gp) - ref).abs() > eb).any()), "%s: bound cannot see a missing K slice" % tag
    return "[%s, conv %s] max(err/bound) %.3g  rms(err/bound) %.3g" % (tag, kern, mx, rms)


def test_network_layers(cuda, capfd, monkeypatch):
    """Every convolution of the FFDNet (colour, gray, IPOL, 3xTF32), DDnet and FastDVDnet engines (fp32 training layers
    and the fp16 inference forms, 64-byte rows on and off), one ragged forward launch each."""
    g = torch.Generator().manual_seed(2024)
    report = []                                        # printed at the end: capfd takes everything printed before
    for name, eng in _network_engines(monkeypatch):
        if name.startswith("fastdvdnet"):
            monkeypatch.setenv("SCI_CONV_SW64", "1" if eng.sw64 else "0")
        eng.prepare()
        layers = list(eng.layers) + list(getattr(eng, "layers_inf", None) or [])
        report += [_layer_check(L, cuda, g, "%s layer %d" % (name, i), capfd) for i, L in enumerate(layers)]
        monkeypatch.delenv("SCI_CONV_SW64", raising=False)
    print("\n".join(report))
