"""GPU parity: every HBM-bound kernel, through the C ABI, against the oracle and the golden vectors.

Tolerances (BASELINE.json north_star): index remaps / Bayer / mask handling bit-exact; A, At, projection,
TV within 1e-5 relative (fp32)."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")
REL = 1e-5


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-30))


def _planar_to_stack4(cube, H, W, B):
    """device planar [B,H,W] -> numpy reference stack [h,w,B,4]"""
    from oracle import sci_ops
    from adaptivepnp_sci_b200 import ops
    hwb = ops.planar_to_pixlast(cube, 1, B).view(H, W, B).cpu()
    return sci_ops.oneCh2FourCh(hwb).numpy()


def _stack4_to_planar(stack4, dev):
    from oracle import sci_ops
    from adaptivepnp_sci_b200 import ops
    hwb = sci_ops.fourCh2OneCh(torch.from_numpy(np.ascontiguousarray(stack4))).contiguous().to(dev)
    H, W, B = hwb.shape
    return ops.pixlast_to_planar(hwb, 1, B).view(B, H, W)


def test_remaps_bit_exact(cuda):
    from adaptivepnp_sci_b200 import ops, utils_image as ui
    from oracle import sci_ops
    g = torch.Generator().manual_seed(0)
    for (P, C, B) in [(64 * 3 + 5, 1, 8), (100, 3, 8), (77, 3, 24), (33, 1, 1)]:
        x = torch.rand(P, C, B, generator=g)
        y = ops.pixlast_to_planar(x.to(cuda), C, B)
        assert torch.equal(y.cpu(), x.permute(2, 1, 0).contiguous())
        assert torch.equal(ops.planar_to_pixlast(y, C, B).cpu(), x)
    d = np.load(os.path.join(G, "operators.npz"))
    theta = torch.from_numpy(d["theta"]).to(cuda)
    one = ui.fourCh2OneCh(theta)
    assert np.array_equal(one.cpu().numpy(), d["merge"])
    assert np.array_equal(ui.oneCh2FourCh(one).cpu().numpy(), d["theta"])
    y4 = torch.rand(8, 6, 4, generator=g)
    assert torch.equal(ui.fourCh2OneCh(y4.to(cuda)).cpu(), sci_ops.fourCh2OneCh(y4))
    assert torch.equal(ui.oneCh2ThreeCh(one).cpu(), sci_ops.oneCh2ThreeCh(one.cpu()))
    rgb = torch.from_numpy(d["rgb"]).to(cuda)
    assert np.array_equal(ui.gen_bayer_img(rgb, 4).cpu().numpy(), d["rgb_to_bayer4"])
    assert torch.equal(ui.gen_bayer_img(rgb, 1).cpu(), sci_ops.gen_bayer_img(rgb.cpu(), 1))
    for a, b in zip(ui.masks_CFA_Bayer_tensor((6, 8)), sci_ops.masks_CFA_Bayer_tensor((6, 8))):
        assert torch.equal(a.cpu(), b)


def test_split_init_and_operators(cuda):
    from adaptivepnp_sci_b200 import ops, utilspy
    from oracle import sci_ops
    d = np.load(os.path.join(G, "operators.npz"))
    y, Phi = torch.from_numpy(d["meas"]).to(cuda), torch.from_numpy(d["mask"]).to(cuda)
    H, W, B = Phi.shape
    phi, phisum, theta0 = ops.bayer_split_init(y, Phi, None)
    # mask handling bit-exact, incl. Phi_sum == 0 -> 1
    assert torch.equal(phi.cpu(), Phi.cpu().permute(2, 0, 1).contiguous())
    assert np.array_equal(sci_ops.oneCh2FourCh(phisum.cpu().unsqueeze(2)).numpy()[:, :, 0, :], d["Phi_sum"])
    assert np.array_equal(_planar_to_stack4(theta0, H, W, B), d["x0_At"])          # binary mask: y*phi exact
    warm = torch.rand(H, W, B).to(cuda)
    _, _, th_w = ops.bayer_split_init(y, Phi, warm)
    assert torch.equal(th_w.cpu(), warm.cpu().permute(2, 0, 1).contiguous())
    # A_/At_ on strided Bayer-phase views, reference signatures
    theta = torch.from_numpy(d["theta"]).to(cuda)
    yall, Phiall, _, _ = (t.to(cuda) for t in sci_ops.bayer_split_init(y.cpu(), Phi.cpu(), None))
    for ib in range(4):
        assert _rel(utilspy.A_(theta[..., ib], Phiall[..., ib]).cpu(), d["A"][..., ib]) < REL
        assert _rel(utilspy.At_(yall[..., ib], Phiall[..., ib]).cpu(), d["At"][..., ib]) < REL


@pytest.mark.parametrize("B", [8, 6, 24])
def test_projection(cuda, B):
    """vectorised (B=8), generic (B=6) and large-scale frame count (B=24) paths vs the oracle; B=8 also vs golden."""
    from adaptivepnp_sci_b200 import ops
    from oracle import sci_ops, synthetic
    if B == 8:
        d = np.load(os.path.join(G, "operators.npz"))
        meas, mask, theta4, b4 = d["meas"], d["mask"], d["theta"], d["b"]
    else:
        meas, mask, _ = synthetic.make_case(32, 48, B, 5 + B, True)
        g = torch.Generator().manual_seed(B)
        theta4 = torch.rand(16, 24, B, 4, generator=g).numpy()
        b4 = (0.1 * torch.randn(16, 24, B, 4, generator=g)).numpy()
    y, Phi = torch.from_numpy(meas), torch.from_numpy(mask)
    yall, Phiall, Psum, _ = sci_ops.bayer_split_init(y, Phi, None)
    ref1 = sci_ops.project_stage1(torch.from_numpy(theta4), torch.from_numpy(b4), yall, Phiall, Psum, 1, 0.01).numpy()
    ref2 = sci_ops.project_stage2(torch.from_numpy(theta4), torch.from_numpy(b4), yall, Phiall, Psum, 1, 0.55).numpy()
    phi, phisum, _ = ops.bayer_split_init(y.to(cuda), Phi.to(cuda), None)
    H, W, _ = Phi.shape
    theta, b = _stack4_to_planar(theta4, cuda), _stack4_to_planar(b4, cuda)
    x = torch.empty_like(theta)
    ops.project_stage1(theta, b, phi, y.to(cuda), phisum, x, 1, 0.01)
    assert _rel(_planar_to_stack4(x, H, W, B), ref1) < REL
    ops.project_stage2(theta, b, phi, y.to(cuda), phisum, x, 1, 0.55)
    assert _rel(_planar_to_stack4(x, H, W, B), ref2) < REL
    if B == 8:
        assert _rel(ref1, d["proj1"]) == 0 and _rel(ref2, d["proj2"]) == 0
    # fused PSNR accumulation of stage 1
    orig = torch.rand_like(theta)
    sse = torch.zeros(1, dtype=torch.float64, device=cuda)
    ops.project_stage1(theta, b, phi, y.to(cuda), phisum, x, 1, 0.01, orig=orig, sse=sse)
    want = float(((x - orig).double() ** 2).sum())
    assert abs(float(sse) - want) / want < 1e-9


# (100, 76), (34, 130): ragged tiles in both directions; (256, 320): several full tiles; B = 1 .. 8 frames
@pytest.mark.parametrize("shape", [(64, 64, 2), (40, 136, 3), (256, 256, 8), (64, 64, 8), (100, 76, 3), (256, 320, 2),
                                   (34, 130, 1)])
def test_tv_chambolle(cuda, shape):
    """TV prior vs the oracle restatement on ragged tile counts, incl. the early-stop decision per channel."""
    from adaptivepnp_sci_b200 import ops
    from oracle import tv_chambolle
    H, W, B = shape
    rng = np.random.default_rng(H + W)
    yy, xx = np.mgrid[0:H // 2, 0:W // 2]
    B += 1                                         # + one nearly flat frame
    stack = np.empty((H // 2, W // 2, B, 4), np.float32)
    for t in range(B - 1):
        for ib in range(4):
            # large-amplitude channels make the energy converge fast: the reference loop stops at i=3 (sigma 8)
            # or i=1 (sigma 50); ordinary channels run all 5 iterations
            noise = (0.08, 8.0, 50.0)[(t + ib) % 3] * rng.standard_normal((H // 2, W // 2))
            stack[:, :, t, ib] = 0.5 + 0.3 * np.sin((xx + 3 * t) / 9.0) * np.cos((yy + ib) / 7.0) + noise
    stack[:, :, B - 1] = 0.5 + 0.02 * rng.random((H // 2, W // 2, 4))
    ref, stops = tv_chambolle.denoise_tv_chambolle(stack.reshape(H // 2, W // 2, 4 * B), 0.1, n_iter_max=5,
                                                   multichannel=True, return_stops=True)
    x = _stack4_to_planar(stack, cuda)
    theta = torch.empty_like(x)
    nstop = torch.zeros(4 * B, dtype=torch.int32, device=cuda)
    ws = ops.TvWorkspace(H, W, B, cuda)
    ops.tv_chambolle(x, None, 0.0, theta, None, 0.0, False, ws, weight=0.1, n_iter_max=5, nstop_out=nstop)
    got_stops = nstop.cpu().numpy().reshape(B, 4)
    want_stops = np.minimum(np.array(stops).reshape(B, 4), 4)
    assert np.array_equal(got_stops, want_stops), (got_stops, want_stops)
    assert _rel(_planar_to_stack4(theta, H, W, B), ref.reshape(H // 2, W // 2, B, 4)) < REL
    assert (want_stops == 1).any() and (want_stops == 3).any() and (want_stops == 4).any()   # all exits exercised
    # fused form: theta = clip(TV(x + c*b)), b' = b + s*(x - theta)
    b = 0.05 * torch.randn_like(x)
    b2 = torch.empty_like(b)
    nstop.zero_()
    ops.tv_chambolle(x, b, -1.0, theta, b2, -1.0, True, ws, nstop_out=nstop)
    f = (x - b)
    ref2, stops2 = tv_chambolle.denoise_tv_chambolle(_planar_to_stack4(f, H, W, B).reshape(H // 2, W // 2, 4 * B), 0.1,
                                                     n_iter_max=5, multichannel=True, return_stops=True)
    got_stops2 = nstop.cpu().numpy().reshape(B, 4)
    assert np.array_equal(got_stops2, np.minimum(np.array(stops2).reshape(B, 4), 4)), got_stops2
    assert (got_stops2 < 4).any()                  # the fix-up pass rewrote channels that stopped early
    ref2 = np.clip(ref2.reshape(H // 2, W // 2, B, 4), 0, 1)
    assert _rel(_planar_to_stack4(theta, H, W, B), ref2) < REL
    want_b = (b - (x - theta)).cpu()
    assert torch.allclose(b2.cpu(), want_b, atol=1e-7, rtol=0)


def test_malvar_and_dual_update(cuda):
    from adaptivepnp_sci_b200 import ops
    from oracle import demosaic, sci_ops
    d = np.load(os.path.join(G, "operators.npz"))
    # golden: the reference's tensor Malvar on a 20x28 CFA (borders = torch reflect)
    cfa = torch.from_numpy(d["malvar_cfa"]).to(cuda)
    H, W = cfa.shape
    x_rgb = torch.empty((1, 3, H, W), device=cuda)
    ops.malvar2004(cfa.view(1, H, W).contiguous(), None, 0.0, None, 0.0, x_rgb, None)
    got = x_rgb[0].permute(1, 2, 0).cpu().numpy()
    assert _rel(got, d["malvar_rgb"]) < REL
    sites = np.zeros((H, W, 3), bool)              # CFA sites are copied, not filtered: bit-exact there
    sites[0::2, 0::2, 0] = sites[0::2, 1::2, 1] = sites[1::2, 0::2, 1] = sites[1::2, 1::2, 2] = True
    assert np.array_equal(got[sites], d["malvar_rgb"][sites])
    # multi-frame, ragged tiles, fused x + c*b and -w/tau
    g = torch.Generator().manual_seed(9)
    B, H, W = 3, 44, 70
    x = torch.rand(B, H, W, generator=g)
    b = 0.1 * torch.randn(B, H, W, generator=g)
    w = torch.randn(B, 3, H, W, generator=g)
    inv_rou = float(np.float32(1 / 0.55))
    R, Gm, Bm = sci_ops.masks_CFA_Bayer_tensor((H, W))
    m = x + inv_rou * b
    ref = torch.stack([demosaic.malvar2004_tensor(m[t], R, Gm, Bm).permute(2, 0, 1) for t in range(B)])
    x_rgb = torch.empty((B, 3, H, W), device=cuda)
    u = torch.empty_like(x_rgb)
    ops.malvar2004(x.to(cuda), b.to(cuda), inv_rou, w.to(cuda), 1 / 100, x_rgb, u)
    assert _rel(x_rgb.cpu(), ref) < REL
    assert _rel(u.cpu(), ref - (1 / 100) * w) < REL
    # dual update: theta = clip(samples), b += x - theta, w += x_rgb - xhat, PSNR; both first_iter modes
    xhat = torch.rand(B, 3, H, W, generator=g) * 1.4 - 0.2
    orig = torch.rand(B, H, W, generator=g)
    for first in (False, True):
        bb, ww, th = b.clone().to(cuda), w.clone().to(cuda), torch.empty(B, H, W, device=cuda)
        sse = torch.zeros(1, dtype=torch.float64, device=cuda)
        ops.dual_update_rgb(xhat.to(cuda), ref.to(cuda), ww, x.to(cuda), bb, th, first, orig=orig.to(cuda), sse=sse)
        samp = sci_ops.fourCh2OneCh(sci_ops.rgb_to_bayer4(xhat.permute(2, 3, 1, 0))).permute(2, 0, 1)
        th_ref = samp.clip(0, 1)
        assert torch.equal(th.cpu(), th_ref)                               # Bayer indexing + clip bit-exact
        x_eff = samp if first else x
        assert torch.equal(bb.cpu(), b + (x_eff - th_ref))
        assert torch.equal(ww.cpu(), w + (ref - xhat))
        want = float(((th_ref - orig).double() ** 2).sum())
        assert abs(float(sse) - want) / want < 1e-6
    assert torch.equal(ops.rgb_to_bayer(xhat.to(cuda)).cpu(), samp)
    assert torch.equal(ops.bayer_to_rgb_sparse(x.to(cuda)).cpu(), sci_ops.oneCh2ThreeCh(x.permute(1, 2, 0)).permute(3, 2, 0, 1))


def test_psnr_accum(cuda):
    from adaptivepnp_sci_b200 import iqa, ops
    from oracle import iqa as oiqa
    g = torch.Generator().manual_seed(4)
    a, o = torch.rand(5, 40, 52, generator=g), torch.rand(5, 40, 52, generator=g)
    sse = torch.zeros(5, dtype=torch.float64, device=cuda)
    ops.psnr_accum(a.to(cuda), o.to(cuda), sse)
    got = iqa.psnr_from_sse(sse.cpu().numpy(), 40 * 52)
    for t in range(5):
        assert abs(got[t] - oiqa.compare_psnr(o[t].numpy(), a[t].numpy(), 1.)) < 1e-9
    assert abs(iqa.ssim(a[0].numpy(), o[0].numpy()) - oiqa.compare_ssim(a[0].numpy(), o[0].numpy())) < 1e-12


def test_ssim_on_device_matches_oracle(cuda):
    """sci_ssim_accum (SURVEY §8(f).4) against the oracle's restatement of skimage's structural_similarity (float64)."""
    from adaptivepnp_sci_b200 import ops
    from oracle import iqa, synthetic
    _, _, orig = synthetic.make_case(64, 96, 4, 11, bayer=True)
    rng = np.random.default_rng(3)
    rec = np.clip(orig + 0.05 * rng.standard_normal(orig.shape), 0, 1).astype(np.float32)
    a = torch.from_numpy(rec).permute(2, 0, 1).contiguous().cuda()
    o = torch.from_numpy(orig).permute(2, 0, 1).contiguous().cuda()
    got = ops.ssim_frames(a, o).cpu().numpy()
    want = np.array([iqa.compare_ssim(orig[:, :, t], rec[:, :, t], data_range=1.) for t in range(4)])
    assert np.max(np.abs(got - want)) < 1e-10
