"""Tiled == un-tiled on REAL GPUs (one strip per GPU, NCCL process group, P2P halo stores over NVLink), tensor-core engine.

    torchrun --nproc-per-node N tools/check_tiled_multi_gpu.py [--size 1024x512x8] [--impl tc] [--deep-demosaic]

Every rank reconstructs its rows of one frame (4 inference iterations + one online update); rank 0 then repeats the
reconstruction un-tiled on its own GPU and prints the differences as one JSON line.  ``--deep-demosaic``: DDnet (synthetic
weights) on the strips instead of Malvar."""
import argparse, io, json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
ap = argparse.ArgumentParser()
ap.add_argument("--size", default="1024x512x8")
ap.add_argument("--impl", default="tc")
ap.add_argument("--deep-demosaic", action="store_true")
a = ap.parse_args()
os.environ["SCI_CONV_IMPL"] = a.impl
import numpy as np, torch
from adaptivepnp_sci_b200 import parallel
from adaptivepnp_sci_b200.dvp_linear_inv_2_stage_ADMM_tensor_online import twoStageAdmm_denoise_bayer
from adaptivepnp_sci_b200.fastdvdnet_adapter import DataParallelLike
from adaptivepnp_sci_b200.fastdvdnet_models import FastDVDnet
from adaptivepnp_sci_b200.network_demosaicking import DDnet
from adaptivepnp_sci_b200.synthetic import ddnet_synthetic_state_dict, fastdvdnet_synthetic_state_dict, make_case
from adaptivepnp_sci_b200.utilspy import worker_init_fn

H, W, B = (int(v) for v in a.size.split("x"))
ctx = parallel.init()
tile = parallel.TileContext(ctx, H, W)
meas, mask, orig = make_case(H, W, B, 515, bayer=True)
warm = np.clip(meas[:, :, None] * mask / np.maximum(mask.sum(2, keepdims=True), 1), 0, 1).astype(np.float32)
KW = dict(show_iqa=True, demosaic_method='malvar2004', lr_=2e-6, interval_iter=3, update_=True, update_per_iter=1, update_times=-1)


def model():
    m = DataParallelLike(FastDVDnet())
    m.load_state_dict({"module." + k: v for k, v in fastdvdnet_synthetic_state_dict().items()}, strict=True)
    return m.eval().cuda()


def demosaicker():
    if not a.deep_demosaic:
        return None
    dm = DDnet()
    dm.load_state_dict(ddnet_synthetic_state_dict(), strict=True)
    return dm.eval().cuda()


KW["model_demosaic"] = demosaicker()
m = model()
worker_init_fn(0)
sl = tile.slice_rows
r = twoStageAdmm_denoise_bayer(sl(meas), sl(mask), 1, 0.01, 'fastdvd_color', [5], False, [12 / 255],
                               x0_bayer=torch.from_numpy(sl(warm)).cuda(), X_orig=sl(orig), model_denoise=m, logf=io.StringIO(),
                               tile=tile, **KW)
used_p2p = tile.p2p is not None
w_t = m.state_dict()["module.temp2.inc.convblock.3.weight"].cpu().numpy()
ctx.barrier()
if ctx.rank == 0:
    m2 = model()
    worker_init_fn(0)
    ref = twoStageAdmm_denoise_bayer(meas, mask, 1, 0.01, 'fastdvd_color', [5], False, [12 / 255],
                                     x0_bayer=torch.from_numpy(warm).cuda(), X_orig=orig, model_denoise=m2, logf=io.StringIO(), **KW)
    w_r = m2.state_dict()["module.temp2.inc.convblock.3.weight"].cpu().numpy()
    print(json.dumps({"n_gpus": ctx.world, "size": a.size, "impl": a.impl, "p2p_halo_exchange": used_p2p,
                      "demosaic": "ddnet" if a.deep_demosaic else "malvar",
                      "max_abs_rgb": float(np.max(np.abs(r[0] - ref[0]))), "max_abs_bayer": float(np.max(np.abs(r[1] - ref[1]))),
                      "max_abs_psnr_all": float(np.max(np.abs(np.array(r[4]) - np.array(ref[4])))),
                      "max_abs_weight": float(np.max(np.abs(w_t - w_r))), "mean_abs_weight": float(np.mean(np.abs(w_t - w_r))),
                      "halo_bytes_per_rank": tile.halo_bytes_moved}))
ctx.barrier()
ctx.finalize()
