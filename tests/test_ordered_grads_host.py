"""CPU: workspace sizes of the fixed-order backward reductions, and the argument checks of their calls.

The ordered weight gradient, fused column sums and act_bwd column sums store one partial per CTA into a slot of a
caller-provided workspace and add the slots in slot order.  The size queries are host arithmetic on the launch plan, and
a missing or too-small workspace is refused before anything touches the GPU - so all of it is checked here without one."""
import ctypes

import pytest

SCI_EINVAL = -1
FAKE = 1 << 20                       # a 16-byte aligned non-NULL address: never dereferenced by the checks below


def _L():
    from adaptivepnp_sci_b200 import _lib
    return _lib


def _wgrad_bytes(Ci, Co, s, N, H, W, impl=0):
    from adaptivepnp_sci_b200 import engine
    d = engine.WgradDesc(FAKE, FAKE, None, FAKE, N, H, W, Ci, Co, s)
    return _L().lib.sci_conv3x3_wgrad_workspace_bytes(ctypes.byref(d), impl)


def _tiles(N, H, W, s):
    return N * -(-((H - 1) // s + 1) // 8) * -(-((W - 1) // s + 1) // 8)


@pytest.mark.parametrize("Ci,Co,s,N,H,W", [(32, 64, 1, 2, 37, 300), (64, 64, 1, 1, 8, 8), (96, 32, 1, 8, 512, 512),
                                           (32, 32, 1, 1, 20, 20)])
def test_wgrad_v3_slots(Ci, Co, s, N, H, W):
    assert _wgrad_bytes(Ci, Co, s, N, H, W) == min(_tiles(N, H, W, s), 148) * 9 * Co * Ci * 4


@pytest.mark.parametrize("Ci,Co,s,N,H,W,m_tiles", [(128, 128, 1, 8, 128, 128, 1), (128, 256, 1, 8, 128, 128, 2),
                                                   (64, 128, 2, 2, 37, 301, 1), (32, 256, 2, 2, 37, 301, 2),
                                                   (128, 64, 1, 1, 16, 16, 1), (64, 128, 1, 1, 8, 8, 1)])
def test_wgrad_v2_slots(Ci, Co, s, N, H, W, m_tiles):
    assert _wgrad_bytes(Ci, Co, s, N, H, W) == max(1, min(_tiles(N, H, W, s), 148 // (3 * m_tiles))) * 9 * Co * Ci * 4


def test_wgrad_reference_slots():
    # fp32 reference kernel: pixel chunks of at least 256 pixels, at most 2 per SM, rounded to 16-pixel steps
    npix = 2 * 37 * 300
    chunks = min(296, -(-npix // 256))
    ppb = -(-(-(-npix // chunks)) // 16) * 16
    assert _wgrad_bytes(32, 64, 1, 2, 37, 300, impl=1) == -(-npix // ppb) * 9 * 64 * 32 * 4
    assert _wgrad_bytes(32, 64, 1, 8, 512, 512, impl=1) == 296 * 9 * 64 * 32 * 4


def test_wgrad_unsupported_shape_needs_nothing():
    assert _wgrad_bytes(40, 20, 1, 1, 16, 16, impl=0) == 0        # tensor-core kernels: channels % 32
    assert _wgrad_bytes(40, 20, 1, 1, 16, 16, impl=1) > 0


def test_headline_workspace_sizes():
    """FastDVDnet at 8 x 512 x 512: the slot sets of the 32 layers of one backward add up to 615 MB (154 M floats); the
    largest single layer, 128->128 at 128 x 128 with 49 slots, is 29 MB - the size the engine's one scratch buffer grows
    to.  Colour FFDNet at 8 x 512 x 512 (12 layers at 256 x 256): 195 MB."""
    from adaptivepnp_sci_b200 import engine
    from adaptivepnp_sci_b200.fastdvdnet_models import FastDVDnet
    from adaptivepnp_sci_b200.network_ffdnet import FFDNet
    e = engine.FastDVDnetEngine(FastDVDnet(num_input_frames=5))
    level = [0, 0, 0, 1, 1, 1, 2, 2, 2, 2, 2, 1, 1, 1, 0, 0]        # input resolution of each DenBlock conv: 512 >> level
    sizes = [_wgrad_bytes(L.Ci_pad, L.Co_pad, L.stride, 8, 512 >> lv, 512 >> lv) for L, lv in zip(e.t1.L, level)]
    assert all(b > 0 for b in sizes)
    total = 2 * sum(sizes)                                           # two DenBlocks of the same shapes
    assert 153.5e6 < total / 4 < 154e6 and 614e6 < total < 616e6
    assert max(sizes) == 49 * 9 * 128 * 128 * 4 and 28.8e6 < max(sizes) < 29e6
    f = engine.FFDNetEngine(FFDNet(3, 3, 96, 12, 'R'))
    ffd = sum(_wgrad_bytes(L.Ci_pad, L.Co_pad, 1, 8, 256, 256) for L in f.layers)
    assert 195e6 < ffd < 196e6


@pytest.mark.parametrize("n_pix,C", [(22200, 48), (3001, 256), (777, 32), (8 * 512 * 512, 96), (1, 1)])
def test_act_bwd_slots(n_pix, C):
    rows = max(1, 256 // C)
    assert _L().lib.sci_act_bwd_workspace_bytes(n_pix, C) == min(148 * 8, -(-n_pix // rows)) * 2 * C * 4


def _colsum_desc(Cin, Cout, ps, N, H, W, s2=True, mask=True):
    from adaptivepnp_sci_b200 import engine
    d = engine.ConvDesc()
    for k, v in dict(x=FAKE, w=FAKE, y=FAKE, N=N, H=H, W=W, Cin=Cin, Cout=Cout, stride=1, pixel_shuffle=ps, round_tf32=1,
                     mask_y=FAKE if mask else None, col_s1=FAKE, col_s2=FAKE if s2 else None, mask_relu=1).items():
        setattr(d, k, v)
    return d


@pytest.mark.parametrize("Cin,Cout,ps,launches", [(64, 64, 0, 1), (32, 32, 0, 1), (64, 128, 1, 1), (128, 256, 1, 2)])
def test_fused_column_sum_slots(Cin, Cout, ps, launches):
    lib = _L().lib
    ncol = Cout // 4 if ps else Cout
    # a large image: every launch has 148 CTAs, one slot [col_s1 | col_s2] of the stored channels each
    d = _colsum_desc(Cin, Cout, ps, 8, 512, 512)
    assert lib.sci_conv3x3_fwd_workspace_bytes(ctypes.byref(d), 0) == launches * 148 * 2 * ncol * 4
    small = _colsum_desc(Cin, Cout, ps, 1, 4, 20)
    b = lib.sci_conv3x3_fwd_workspace_bytes(ctypes.byref(small), 0)
    assert 0 < b < launches * 148 * 2 * ncol * 4 and b % (launches * 2 * ncol * 4) == 0
    # no column sums, no fused mask or the fp32 reference engine: nothing to order
    d.col_s1 = d.col_s2 = None
    assert lib.sci_conv3x3_fwd_workspace_bytes(ctypes.byref(d), 0) == 0
    assert lib.sci_conv3x3_fwd_workspace_bytes(ctypes.byref(_colsum_desc(Cin, Cout, ps, 8, 64, 64, mask=False)), 0) == 0
    assert lib.sci_conv3x3_fwd_workspace_bytes(ctypes.byref(_colsum_desc(Cin, Cout, ps, 8, 64, 64)), 1) == 0


def test_ordered_calls_refuse_missing_or_small_workspace():
    """Refused with SCI_EINVAL before any launch: these calls never reach the GPU."""
    from adaptivepnp_sci_b200 import engine
    lib = _L().lib
    # act_bwd
    nb = lib.sci_act_bwd_workspace_bytes(22200, 48)
    assert lib.sci_act_bwd_ordered(FAKE, FAKE, FAKE, 22200, 48, 1, FAKE, FAKE, None, nb, None) == SCI_EINVAL
    assert lib.sci_act_bwd_ordered(FAKE, FAKE, FAKE, 22200, 48, 1, FAKE, FAKE, FAKE, nb - 4, None) == SCI_EINVAL
    assert lib.sci_act_bwd_ordered(FAKE, FAKE, FAKE, 22200, 48, 1, FAKE, FAKE, FAKE + 4, nb, None) == SCI_EINVAL
    assert b"workspace" in lib.sci_last_error()
    # weight gradient, both engines
    for impl in (0, 1):
        d = engine.WgradDesc(FAKE, FAKE, None, FAKE, 2, 37, 300, 32, 64, 1)
        need = lib.sci_conv3x3_wgrad_workspace_bytes(ctypes.byref(d), impl)
        d.workspace, d.workspace_bytes = FAKE, need - 4
        assert lib.sci_conv3x3_wgrad(ctypes.byref(d), impl, None) == SCI_EINVAL
        d.workspace, d.workspace_bytes = None, need
        assert lib.sci_conv3x3_wgrad(ctypes.byref(d), impl, None) == SCI_EINVAL
    # fused column sums
    d = _colsum_desc(64, 64, 0, 2, 37, 300)
    need = lib.sci_conv3x3_fwd_workspace_bytes(ctypes.byref(d), 0)
    d.workspace, d.workspace_bytes = FAKE, need - 8
    assert lib.sci_conv3x3_dgrad(ctypes.byref(d), 0, None) == SCI_EINVAL
    d.workspace, d.workspace_bytes = None, need
    assert lib.sci_conv3x3_dgrad(ctypes.byref(d), 0, None) == SCI_EINVAL
