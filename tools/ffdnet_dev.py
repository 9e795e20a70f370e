"""Where does the FFDNet tensor-core engine deviate from the fp32 engine at 512x512x8 (config 3): inference or fine-tune?"""
import io, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from adaptivepnp_sci_b200.dvp_linear_inv_2_stage_ADMM_tensor_online import admm_denoise_bayer_demosaic_pre, twoStageAdmm_denoise_bayer
from adaptivepnp_sci_b200.network_ffdnet import FFDNet
from adaptivepnp_sci_b200.synthetic import make_case
from adaptivepnp_sci_b200.utilspy import worker_init_fn
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
meas, mask, orig = make_case(512, 512, 8, 3000, bayer=True)
warm = admm_denoise_bayer_demosaic_pre(meas, mask, 1, 0.01, 'tv', [40], False, [0], X_orig=None, show_iqa=False)[0]
g = np.load(os.path.join(ROOT, "tests", "golden", "fullsize.npz"))
res = {}
for upd in (False, True):
    for impl in ("ref", "tc"):
        os.environ["SCI_CONV_IMPL"] = impl
        m = FFDNet(3, 3, 96, 12, 'R'); m.load_state_dict(torch.load(os.path.join(ROOT, "model_zoo", "ffdnet_color.pth"))); m = m.eval().cuda()
        worker_init_fn(0)
        r = twoStageAdmm_denoise_bayer(meas, mask, 1, 0.01, 'ffdnet_color', [6, 6, 4], False, [25 / 255, 12 / 255, 6 / 255],
                                       x0_bayer=torch.from_numpy(warm).cuda(), X_orig=orig, model_denoise=m, show_iqa=True,
                                       lr_=2e-6, interval_iter=6, logf=io.StringIO(), update_=upd, update_per_iter=2)
        res[(upd, impl)] = r[1]
        del m; torch.cuda.empty_cache()
    d = np.abs(res[(upd, "tc")] - res[(upd, "ref")])
    print("update=%s: tc vs fp32 engine max-abs %.3e  mean-abs %.3e" % (upd, d.max(), d.mean()))
print("fp32 engine (update) vs reference golden sample: %.3e" % np.abs(res[(True, "ref")][::3, ::3] - g["c3_x_s"]).max())
print("tc engine   (update) vs reference golden sample: %.3e" % np.abs(res[(True, "tc")][::3, ::3] - g["c3_x_s"]).max())

os.environ["SCI_CONV_IMPL"] = "tc"
m = FFDNet(3, 3, 96, 12, 'R'); m.load_state_dict(torch.load(os.path.join(ROOT, "model_zoo", "ffdnet_color.pth"))); m = m.eval().cuda()
u = torch.rand(8, 3, 512, 512, device="cuda")
eng = m.engine()
for _ in range(3):
    eng.forward(u, 12 / 255)
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record()
for _ in range(20):
    eng.forward(u, 12 / 255)
b.record(); torch.cuda.synchronize()
print("FFDNet-colour inference pass 8x512x512: %.3f ms" % (a.elapsed_time(b) / 20))
