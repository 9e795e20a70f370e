"""GPU: grayscale FastDVDnet on single-plane boundary kernels ('fastdvd_gray').

Every planes = 1 boundary kernel against the planes = 3 kernel on the zero-embedded cube, bit for bit; the engine on gray
frames against its run on the embedded cube; one fine-tune call and the whole derived loop against the derived oracle
(oracle.gray_fastdvd: "parity vs derived oracle")."""
import io

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from test_gpu_conv import _fastdvd, impl  # noqa: E402,F401

TOL = {"ref": 2e-4, "tc": 1e-3}
SIZES = [(16, 16, 3), (40, 52, 5)]


def _bits(t):
    return t.detach().contiguous().cpu().numpy().view(np.uint32)


def _same(a, b):
    assert a.shape == b.shape and np.array_equal(_bits(a), _bits(b))


def _embed(g):
    """[B,1,H,W] -> the zero-embedded colour cube [B,3,H,W] (planes 1 and 2 +0)."""
    e = torch.zeros((g.shape[0], 3) + tuple(g.shape[2:]), dtype=g.dtype, device=g.device)
    e[:, 0:1] = g
    return e


def _gray_model(dev):
    from adaptivepnp_sci_b200.fastdvdnet_adapter import DataParallelLike
    from adaptivepnp_sci_b200.fastdvdnet_models import FastDVDnet
    from adaptivepnp_sci_b200.synthetic import fastdvdnet_gray_synthetic_state_dict
    m = DataParallelLike(FastDVDnet(num_input_frames=5, num_color_channels=1))
    m.load_state_dict({"module." + k: v for k, v in fastdvdnet_gray_synthetic_state_dict().items()}, strict=True)
    return m.eval().to(dev)


def _oracle_gray_model():
    from oracle import networks, synthetic
    m = networks.Wrapped(networks.FastDVDnet(5, 1))
    m.load_state_dict({"module." + k: v for k, v in synthetic.fastdvdnet_gray_synthetic_state_dict().items()}, strict=True)
    return m.eval()


def _twin_zero_entries(net):
    """Every entry of the colour-shaped twin that the embedding of the gray weights sets to zero."""
    twin = net._twin[0]
    out = []
    for blk in (twin.temp1, twin.temp2):
        out.append(blk.inc.convblock[0].weight.detach()[:, 1:3])
        out.append(blk.outc.convblock[3].weight.detach()[1:3])
    return out


# ---- 1. boundary kernels ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("H,W,B", SIZES)
def test_boundary_kernels_one_plane_vs_embedding(cuda, impl, H, W, B):
    from adaptivepnp_sci_b200._lib import call, ptr, stream
    g = torch.Generator(device="cpu").manual_seed(H * W + B)
    frames = torch.rand((B, 1, H, W), generator=g).to(cuda)
    f3 = _embed(frames)
    sigma = 12 / 255
    for rt, cpad in ((1, 32), (0, 32), (0, 16), (1, 48)):       # TF32 split (hi + remainder) and plain fp32 packers
        a1 = torch.full((B, H, W, cpad), 7.0, device=cuda)
        a3 = torch.full((B, H, W, cpad), 7.0, device=cuda)
        call("sci_fastdvd_pack_input_planes", ptr(frames), sigma, ptr(a1), B, 1, H, W, cpad, rt, stream())
        call("sci_fastdvd_pack_input", ptr(f3), sigma, ptr(a3), B, H, W, cpad, rt, stream())
        _same(a1, a3)
    for c in (32, 64):                                           # fp16 packer, both row widths
        h1 = torch.full((B, H, W, c), 3.0, dtype=torch.float16, device=cuda)
        h3 = torch.full((B, H, W, c), 3.0, dtype=torch.float16, device=cuda)
        call("sci_fastdvd_pack_input_half_planes", ptr(frames), sigma, ptr(h1), B, 1, H, W, c, stream())
        call("sci_fastdvd_pack_input_half", ptr(f3), sigma, ptr(h3), B, H, W, c, stream())
        assert np.array_equal(h1.cpu().numpy().view(np.uint16), h3.cpu().numpy().view(np.uint16))
    for cpad in (32, 64):
        y = torch.randn((B, H, W, cpad), generator=g).to(cuda)
        o1, o3 = torch.empty_like(frames), torch.empty_like(f3)
        call("sci_fastdvd_output_planes", ptr(frames), ptr(y), ptr(o1), B, 1, H, W, cpad, stream())
        call("sci_fastdvd_output", ptr(f3), ptr(y), ptr(o3), B, H, W, cpad, stream())
        _same(o1, o3[:, 0:1])
        dout = torch.randn((B, 1, H, W), generator=g).to(cuda)
        d1 = torch.full((B, H, W, cpad), 5.0, device=cuda)
        d3 = torch.full((B, H, W, cpad), 5.0, device=cuda)
        call("sci_fastdvd_output_grad_planes", ptr(dout), ptr(d1), B, 1, H, W, cpad, stream())
        call("sci_fastdvd_output_grad", ptr(_embed(dout)), ptr(d3), B, H, W, cpad, stream())
        _same(d1, d3)
    din = torch.randn((B, H, W, 32), generator=g).to(cuda)
    for acc in (0, 1):
        base = torch.randn((B, 1, H, W), generator=g).to(cuda)
        r1, r3 = base.clone(), _embed(base)
        call("sci_fastdvd_pack_input_grad_planes", ptr(din), ptr(r1), B, 1, H, W, 32, acc, stream())
        call("sci_fastdvd_pack_input_grad", ptr(din), ptr(r3), B, H, W, 32, acc, stream())
        _same(r1, r3[:, 0:1])


@pytest.mark.parametrize("H,W,B", SIZES)
def test_fused_planar_epilogue_one_plane(cuda, impl, H, W, B):
    """The last conv of a DenBlock with the fused `out = in1 - conv` epilogue (tensor-core kernels only): planar_planes = 1
    against plane 0 of planar_planes = 3, on the TF32 training layer and on the fp16 inference chain."""
    if impl != "tc":
        pytest.skip("the fused planar epilogue exists on the tensor-core kernels only")
    net = _gray_model(cuda).module
    eng = net.engine()
    eng.prepare(training=True)
    g = torch.Generator(device="cpu").manual_seed(B)
    in1 = torch.rand((B, 1, H, W), generator=g).to(cuda)
    x = torch.randn((B, H, W, 32), generator=g).to(cuda)
    L = eng.t2.L[15]
    o1, o3 = torch.full_like(in1, 9.0), torch.full((B, 3, H, W), 9.0, device=cuda)
    eng.conv(L, x, B, H, W, None, round_out=False, planar=(in1, o1))
    eng.conv(L, x, B, H, W, None, round_out=False, planar=(_embed(in1), o3))
    _same(o1, o3[:, 0:1])
    assert eng.half
    Lh = eng.t2h[15]
    xh = x[..., :Lh.cin_store].half().contiguous()
    o1, o3 = torch.full_like(in1, 9.0), torch.full((B, 3, H, W), 9.0, device=cuda)
    eng.conv_h(Lh, xh, B, H, W, None, planar=(in1, o1))
    eng.conv_h(Lh, xh, B, H, W, None, planar=(_embed(in1), o3))
    _same(o1, o3[:, 0:1])


# ---- 2. engine ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("H,W,B", [(40, 52, 5), (64, 64, 8)])
def test_engine_gray_vs_embedding(cuda, impl, H, W, B):
    """Inference (fp16 chain on the tensor-core path) and the training forward on [B,1,H,W] equal plane 0 of the twin's run
    on the embedded cube bit for bit; the backward pass leaves every embedded zero of the twin with a zero gradient."""
    net = _gray_model(cuda).module
    eng = net.engine()
    g = torch.Generator(device="cpu").manual_seed(H + B)
    v = torch.rand((B, 1, H, W), generator=g).to(cuda)
    for train in (False, True):
        got = eng.forward(v, 12 / 255, train=train).clone()
        want = eng.forward(_embed(v), 12 / 255, train=train).clone()
        assert got.shape == (B, 1, H, W)
        _same(got, want[:, 0:1])
    dout = torch.randn((B, 1, H, W), generator=g).to(cuda)
    eng.forward(v, 12 / 255, train=True)
    eng.backward(dout)
    grads = [eng.bucket.grad_view(p) for p in (net._twin[0].temp1.inc.convblock[0].weight,
                                                 net._twin[0].temp2.inc.convblock[0].weight)]
    assert all(float(t[:, 1:3].abs().max()) == 0.0 for t in grads)
    assert all(float(t[:, 0].abs().max()) > 0.0 for t in grads)
    gout = [eng.bucket.grad_view(b.outc.convblock[3].weight) for b in (net._twin[0].temp1, net._twin[0].temp2)]
    assert all(float(t[1:3].abs().max()) == 0.0 and float(t[0].abs().max()) > 0.0 for t in gout)


def test_frame_wise_gray_adapter_vs_embedding(cuda, impl):
    """fastdvdnet_denoiser(gray=True) (single-plane path, reflect pad to x4) returns the bits of the embedded path."""
    from adaptivepnp_sci_b200 import ops
    from adaptivepnp_sci_b200.fastdvdnet_adapter import fastdvdnet_denoiser
    m = _gray_model(cuda)
    rs = np.random.RandomState(4)
    vn = rs.rand(38, 50, 6).astype(np.float32)                    # [H,W,F], not multiples of 4
    got = fastdvdnet_denoiser(vn, 20 / 255, model=m, gray=True)
    seq = torch.from_numpy(vn).cuda().permute(2, 0, 1).unsqueeze(1).contiguous()
    padded, H, W = ops.pad_to_multiple(_embed(seq), 4)
    want = ops.crop_to(m.module.engine().forward(padded, 20 / 255, train=False), H, W)[:, 0].permute(1, 2, 0)
    assert got.shape == vn.shape
    assert np.array_equal(got.view(np.uint32), want.contiguous().cpu().numpy().view(np.uint32))


# ---- 3. one fine-tune call ---------------------------------------------------------------------------------------------
def _finetune_case(cuda):
    from oracle import synthetic
    H, W, B = 64, 64, 8
    meas, mask, orig = synthetic.make_case(H, W, B, 1001, bayer=False)
    x = np.clip(orig + np.random.RandomState(2).normal(0, 0.05, orig.shape), 0, 1).astype(np.float32)
    return meas, mask, x


def test_one_finetune_call_vs_derived_oracle(cuda, impl):
    from adaptivepnp_sci_b200.fastdvdnet_adapter import finetune_and_denoise
    from oracle import gray_fastdvd
    meas, mask, x = _finetune_case(cuda)
    H, W, B = x.shape
    lr, steps, sigma = 2e-6, 2, 12 / 255
    mo = _oracle_gray_model()
    sd0 = {k: v.clone() for k, v in mo.module.state_dict().items()}
    np.random.seed(1234)
    ref, _ = gray_fastdvd.fastdvdnet_gray_denoise_full_tensor(torch.from_numpy(x), torch.from_numpy(meas), torch.from_numpy(mask),
                                                          sigma, mo, lr, True, steps)
    st_ref = np.random.get_state()
    m = _gray_model(cuda)
    v = torch.from_numpy(x).cuda().permute(2, 0, 1).unsqueeze(1).contiguous()
    phi = torch.from_numpy(mask).cuda().permute(2, 0, 1).contiguous()
    y = torch.from_numpy(meas).cuda()
    np.random.seed(1234)
    out = finetune_and_denoise(v, phi, y, sigma, m, lr, steps)
    st = np.random.get_state()
    got = out[:, 0].permute(1, 2, 0).cpu().numpy()
    assert out.shape == (B, 1, H, W)
    assert np.max(np.abs(got - ref.numpy())) < TOL[impl]
    # the gray state_dict holds the fine-tuned weights: an update direction that flips under rounding moves a weight by at
    # most 2 lr per Adam step (tests/test_gpu_shared_weights.py)
    want_sd, got_sd = mo.module.state_dict(), m.module.state_dict()
    assert list(got_sd.keys()) == list(want_sd.keys())
    moved = 0.0
    for k, w in want_sd.items():
        gw = got_sd[k].cpu()
        assert np.max(np.abs(gw.numpy() - w.numpy())) <= steps * 2 * lr * 1.01, k
        assert np.mean(np.abs(gw.numpy() - w.numpy())) < (0.1 if impl == "ref" else 0.5) * lr, k
        moved = max(moved, float((gw - sd0[k]).abs().max()))
    assert moved > 1e-7
    for t in _twin_zero_entries(m.module):                        # still +0.0, bit for bit
        assert not np.any(_bits(t))
    assert st[0] == st_ref[0] and np.array_equal(st[1], st_ref[1]) and st[2:] == st_ref[2:]


# ---- 4. the whole derived loop -----------------------------------------------------------------------------------------
_ORACLE = {}


def _loop_case(update_times):
    from oracle import admm, gray_fastdvd, synthetic
    if update_times not in _ORACLE:
        meas, mask, orig = synthetic.make_case(64, 64, 8, 1001, bayer=False)
        warm = admm.admm_denoise_bayer_demosaic_pre(meas, mask, 1, 0.01, 'tv', [40], False, [0], X_orig=orig,
                                                    show_iqa=False)[0]
        np.random.seed(77)
        ref = gray_fastdvd.twoStageAdmm_denoise_gray(meas, mask, 'fastdvd_gray', x0=torch.from_numpy(warm),
                                                     model_denoise=_oracle_gray_model(), update_times=update_times,
                                                     **_loop_kw(orig))
        _ORACLE[update_times] = (meas, mask, orig, warm, ref, np.random.get_state())
    return _ORACLE[update_times]


def _loop_kw(orig):
    return dict(iter_max=[5, 2], sigma=[12 / 255, 6 / 255], X_orig=orig, lr_=2e-6, interval_iter=3, update_=True,
                update_per_iter=2)


@pytest.mark.parametrize("update_times", [-1, 1])
def test_stage2_fastdvd_gray_vs_derived_oracle(cuda, impl, update_times):
    from adaptivepnp_sci_b200.dvp_linear_inv_2_stage_ADMM_tensor_online import twoStageAdmm_denoise_gray
    meas, mask, orig, warm, ref, st_ref = _loop_case(update_times)
    m = _gray_model(cuda)
    sd0 = {k: v.cpu().clone() for k, v in m.module.state_dict().items()}
    np.random.seed(77)
    got = twoStageAdmm_denoise_gray(meas, mask, 'fastdvd_gray', x0=torch.from_numpy(warm).cuda(), model_denoise=m,
                                    logf=io.StringIO(), update_times=update_times, **_loop_kw(orig))
    st = np.random.get_state()
    tol = TOL[impl]
    assert len(got) == 6 and got[0].shape == (64, 64, 8) and got[1].shape == (64, 64, 8)
    assert got[5] is m
    assert np.max(np.abs(got[0] - ref[0])) < tol and np.max(np.abs(got[1] - ref[1])) < tol
    assert len(got[4]) == 7 and np.max(np.abs(np.array(got[4]) - np.array(ref[4]))) < 0.05
    assert max(float((v.cpu() - sd0[k]).abs().max()) for k, v in m.module.state_dict().items()) > 1e-7
    assert st[0] == st_ref[0] and np.array_equal(st[1], st_ref[1]) and st[2:] == st_ref[2:]


# ---- 5. grad_sync ------------------------------------------------------------------------------------------------------
def test_grad_sync_sees_the_twin_bucket(cuda, impl):
    """The hook is called once per Adam step with the twin's flat gradient bucket; an identity hook changes nothing it is
    given.  (Two fine-tune runs are not compared bit for bit: the weight gradients are accumulated with atomics, whose
    order, and so whose last bits, vary from run to run.)"""
    from adaptivepnp_sci_b200.dvp_linear_inv_2_stage_ADMM_tensor_online import twoStageAdmm_denoise_gray
    meas, mask, orig, warm, ref, _ = _loop_case(-1)
    m = _gray_model(cuda)
    seen = []

    def hook(g):
        seen.append((g.data_ptr(), g.numel(), g.clone()))
    np.random.seed(77)
    got = twoStageAdmm_denoise_gray(meas, mask, 'fastdvd_gray', x0=torch.from_numpy(warm).cuda(), model_denoise=m,
                                    logf=io.StringIO(), grad_sync=hook, **_loop_kw(orig))
    bucket = m.module._twin[0].engine().bucket
    assert len(seen) == 2 * 2                                     # two updates (k = 3, 6) of two Adam steps each
    assert all(p == bucket.grad.data_ptr() and n == bucket.grad.numel() for p, n, _ in seen)
    assert all(float(g.abs().max()) > 0 for _, _, g in seen)
    tol = TOL[impl]
    assert np.max(np.abs(got[0] - ref[0])) < tol and np.max(np.abs(got[1] - ref[1])) < tol
