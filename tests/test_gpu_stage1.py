"""GPU parity of the whole stage-1 loop (and the 'tv' branch of stage 2) against the oracle / golden vectors."""
import io
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")


def test_stage1_vs_golden_64(cuda):
    from adaptivepnp_sci_b200.dvp_linear_inv_2_stage_ADMM_tensor_online import admm_denoise_bayer_demosaic_pre
    from oracle import synthetic
    d = np.load(os.path.join(G, "loops.npz"))
    meas, mask, orig = synthetic.make_case(64, 64, 8, 1001, bayer=False)
    log = io.StringIO()
    x, psnr_, ssim_, psnr_all = admm_denoise_bayer_demosaic_pre(meas, mask, 1, 0.01, 'tv', [40], False, [0],
                                                                x0_bayer=None, X_orig=orig, model=None,
                                                                show_iqa=True, logf=log)
    assert x.shape == (64, 64, 8) and x.dtype == np.float32 and len(psnr_all) == 40 and len(psnr_) == 8
    # 40 iterations of feedback: fp32 rounding differences may grow, the early-stop decisions must not flip
    assert np.max(np.abs(x - d["s1_x"])) < 2e-5
    assert np.max(np.abs(np.array(psnr_all) - d["s1_psnr_all"])) < 1e-3
    assert np.max(np.abs(np.array(psnr_) - d["s1_psnr"])) < 1e-3
    assert np.max(np.abs(np.array(ssim_) - d["s1_ssim"])) < 1e-5
    assert "ADMM-TV iteration  40, sigma   0/255, PSNR" in log.getvalue()


def test_stage1_vs_oracle_256(cuda):
    """BASELINE config 1 at full size (256x256x8, 40 iterations) against the oracle run live."""
    from adaptivepnp_sci_b200.dvp_linear_inv_2_stage_ADMM_tensor_online import admm_denoise_bayer_demosaic_pre
    from oracle import admm, synthetic
    meas, mask, orig = synthetic.make_case(256, 256, 8, 1001, bayer=False)
    ref = admm.admm_denoise_bayer_demosaic_pre(meas, mask, 1, 0.01, 'tv', [40], False, [0], X_orig=orig)
    got = admm_denoise_bayer_demosaic_pre(meas, mask, 1, 0.01, 'tv', [40], False, [0], X_orig=orig, logf=io.StringIO())
    assert np.max(np.abs(got[0] - ref[0])) < 5e-5
    assert abs(np.mean(got[1]) - np.mean(ref[1])) < 0.01          # dB
    assert np.max(np.abs(np.array(got[3]) - np.array(ref[3]))) < 1e-2


def test_stage2_tv_branch(cuda):
    from adaptivepnp_sci_b200.dvp_linear_inv_2_stage_ADMM_tensor_online import twoStageAdmm_denoise_bayer
    from oracle import synthetic
    d = np.load(os.path.join(G, "loops.npz"))
    meas, mask, orig = synthetic.make_case(64, 64, 8, 3000, bayer=True)
    r = twoStageAdmm_denoise_bayer(meas, mask, 1, 0.01, 'tv', [6], False, [0],
                                   x0_bayer=torch.from_numpy(d["s2_warm"]).cuda(), X_orig=orig, logf=io.StringIO())
    assert len(r) == 4
    assert np.max(np.abs(r[0] - d["s2tv_x"])) < 1e-5
    assert np.max(np.abs(np.array(r[3]) - d["s2tv_psnr_all"])) < 1e-3
    with pytest.raises(ValueError):
        twoStageAdmm_denoise_bayer(meas, mask, denoiser='bm3d', iter_max=1, sigma=[0])


def test_roundtrip_properties_512(cuda):
    """Size-independent properties at the headline size 512x512x8: projection is idempotent on consistent
    data, A(At(y)) = y*Phi_sum, remap round trip, linearity of A."""
    from adaptivepnp_sci_b200 import ops
    from oracle import synthetic
    meas, mask, orig = synthetic.make_case(512, 512, 8, 3000, bayer=True)
    y, Phi = torch.from_numpy(meas).cuda(), torch.from_numpy(mask).cuda()
    phi, phisum, theta0 = ops.bayer_split_init(y, Phi, None)
    assert torch.equal(ops.planar_to_pixlast(phi, 1, 8).view(512, 512, 8), Phi)
    zero = torch.zeros_like(theta0)
    # the ground truth satisfies y = A(orig): projecting it with gamma -> 0 must leave it unchanged
    og = ops.pixlast_to_planar(torch.from_numpy(orig).cuda(), 1, 8).view(8, 512, 512)
    x = torch.empty_like(og)
    ops.project_stage1(og, zero, phi, y, phisum, x, 1.0, 1e-30)
    assert float((x - og).abs().max()) < 1e-5
    # after one projection of anything the measurement is reproduced: A(x) = y wherever Phi_sum > 0 (gamma -> 0)
    ops.project_stage1(theta0, zero, phi, y, phisum, x, 1.0, 1e-30)
    Ax = (x * phi).sum(0)
    has = (phi.sum(0) > 0)
    assert float(((Ax - y).abs() * has).max()) < 1e-4


@pytest.mark.parametrize("impl", ["ref", "tc"])
def test_stage1_deep_branches_vs_golden(cuda, impl, monkeypatch):
    """Deep branches of admm_denoise_bayer_demosaic_pre ('ffdnet_color' / 'fastdvd_color', dvp...online.py:456-503, :552)
    against the reference's own outputs: warm-started and from x0 = At(y), both conv engines."""
    monkeypatch.setenv("SCI_CONV_IMPL", impl)
    from adaptivepnp_sci_b200.dvp_linear_inv_2_stage_ADMM_tensor_online import admm_denoise_bayer_demosaic_pre, np2tch_cuda
    from adaptivepnp_sci_b200.fastdvdnet_adapter import DataParallelLike
    from adaptivepnp_sci_b200.fastdvdnet_models import FastDVDnet
    from adaptivepnp_sci_b200.network_ffdnet import FFDNet
    from oracle import synthetic
    d = np.load(os.path.join(G, "stage1_deep.npz"))
    warm = np.load(os.path.join(G, "loops.npz"))["s2_warm"]
    meas, mask, orig = synthetic.make_case(64, 64, 8, 3000, bayer=True)

    def ffd():
        m = FFDNet(3, 3, 96, 12, 'R')
        m.load_state_dict(torch.load(os.path.join(ROOT, "model_zoo", "ffdnet_color.pth")), strict=True)
        return m.eval().cuda()

    def fdvd():
        m = DataParallelLike(FastDVDnet())
        m.load_state_dict({"module." + k: v for k, v in synthetic.fastdvdnet_synthetic_state_dict().items()}, strict=True)
        return m.eval().cuda()
    tol = {"ref": 2e-4, "tc": 1e-3}[impl]
    for tag, den, mk, sig, its in (("ffd", 'ffdnet_color', ffd, [25 / 255, 12 / 255], [3, 2]),
                                   ("fdvd", 'fastdvd_color', fdvd, [12 / 255], [4])):
        for wtag in ("", "_cold"):
            m = mk()
            r = admm_denoise_bayer_demosaic_pre(meas, mask, 1, 0.01, den, its, False, sig,
                                                x0_bayer=None if wtag else np2tch_cuda(warm), X_orig=orig, model=m,
                                                show_iqa=True, logf=io.StringIO())
            assert len(r) == 6 and r[5] is m and r[0].shape == (64, 64, 3, 8) and r[1].shape == (64, 64, 8)
            assert np.max(np.abs(r[0] - d[tag + wtag + "_rgb"])) < tol and np.max(np.abs(r[1] - d[tag + wtag + "_x"])) < tol
            assert np.max(np.abs(np.array(r[4]) - d[tag + wtag + "_psnr_all"])) < 0.05
            assert np.max(np.abs(np.array(r[2]) - d[tag + wtag + "_psnr"])) < 0.05
    with pytest.raises(NotImplementedError):
        admm_denoise_bayer_demosaic_pre(meas, mask, 1, 0.01, 'ffdnet_color', [3], False, [25 / 255], model=ffd(), update_=True)
    with pytest.raises(ValueError):
        admm_denoise_bayer_demosaic_pre(meas, mask, 1, 0.01, 'PPP', [3], False, [25 / 255])
