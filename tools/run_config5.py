"""BASELINE config 5: large-scale 2048x2048x24 Bayer frame, FastDVDnet, spatial row strips + halo exchange.

    torchrun --nproc-per-node N tools/run_config5.py [--size 2048] [--frames 24] [--iters 8,2] [--no-update] [--tv-warm-start]
                                                     [--deep-demosaic] [--close-form]

Every rank owns H/N rows; prints one JSON line (rank 0) with ms per ADMM iteration (CUDA events, max over ranks),
the PSNR trajectory and the halo bytes moved per iteration.  Stage 2 starts from a crude At-normalised estimate unless
``--tv-warm-start``: then tiled stage 1 (40 TV iterations, as in configs 1-4 and the reference pipeline) produces the warm
start on the same strips and hands it to stage 2 as a device strip; the crude-start PSNR trajectory is reported beside it.
``--deep-demosaic`` demosaics with DDnet (synthetic weights) on the strips instead of Malvar and reports the DDnet share of
an iteration and its frame chunk; ``--close-form`` runs the closed-form demosaic branch (from the second iteration on).
Peak memory is reported per rank."""
import argparse, io, json, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from adaptivepnp_sci_b200 import parallel
from adaptivepnp_sci_b200.dvp_linear_inv_2_stage_ADMM_tensor_online import (admm_denoise_bayer_demosaic_pre,
                                                                            twoStageAdmm_denoise_bayer)
from adaptivepnp_sci_b200.fastdvdnet_adapter import DataParallelLike
from adaptivepnp_sci_b200.fastdvdnet_models import FastDVDnet
from adaptivepnp_sci_b200.network_demosaicking import DDnet
from adaptivepnp_sci_b200.synthetic import ddnet_synthetic_state_dict, fastdvdnet_synthetic_state_dict, make_case
from adaptivepnp_sci_b200.utilspy import worker_init_fn

ap = argparse.ArgumentParser()
ap.add_argument("--size", type=int, default=2048)
ap.add_argument("--frames", type=int, default=24)
ap.add_argument("--iters", default="8,2")
ap.add_argument("--no-update", action="store_true")
ap.add_argument("--tv-warm-start", action="store_true")
ap.add_argument("--deep-demosaic", action="store_true")
ap.add_argument("--close-form", action="store_true")
a = ap.parse_args()
ctx = parallel.init()
H = W = a.size
B = a.frames
iters = [int(v) for v in a.iters.split(",")]
tile = parallel.TileContext(ctx, H, W)
t0 = time.time()
meas, mask, orig = make_case(H, W, B, 5001, bayer=True)
warm = np.clip(meas[:, :, None] * mask / np.maximum(mask.sum(2, keepdims=True), 1), 0, 1).astype(np.float32)
t_data = time.time() - t0
m = DataParallelLike(FastDVDnet())
m.load_state_dict({"module." + k: v for k, v in fastdvdnet_synthetic_state_dict().items()})
m = m.eval().cuda()
dm = None
if a.deep_demosaic:
    dm = DDnet()
    dm.load_state_dict(ddnet_synthetic_state_dict(), strict=True)
    dm = dm.eval().cuda()
worker_init_fn(0)
sl = tile.slice_rows
args = (sl(meas), sl(mask), 1, 0.01, 'fastdvd_color', iters, False, [12 / 255, 6 / 255][:len(iters)])
kw = dict(x0_bayer=torch.from_numpy(sl(warm)).cuda(), X_orig=sl(orig), model_denoise=m, show_iqa=True, lr_=2e-6,
          interval_iter=9, logf=io.StringIO(), update_=not a.no_update, update_per_iter=2, tile=tile, model_demosaic=dm,
          close_form_demosaic=a.close_form)
ms_stage1 = None
if a.tv_warm_start:
    torch.cuda.synchronize(); ctx.barrier()
    s1, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s1.record()
    x_tv = admm_denoise_bayer_demosaic_pre(sl(meas), sl(mask), 1, 0.01, 'tv', [40], False, [0], tile=tile, return_device=True)
    e1.record(); torch.cuda.synchronize()
    ms_stage1 = s1.elapsed_time(e1)               # first call: includes the peer-to-peer set-up
    kw_crude, kw = kw, dict(kw, x0_bayer=x_tv)


def timed(it_list, update):
    kw2 = dict(kw, X_orig=None, show_iqa=False, update_=update)
    torch.cuda.synchronize(); ctx.barrier()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    twoStageAdmm_denoise_bayer(args[0], args[1], 1, 0.01, 'fastdvd_color', it_list, False, [12 / 255, 6 / 255][:len(it_list)], **kw2)
    e.record(); torch.cuda.synchronize()
    ms = torch.tensor([s.elapsed_time(e)], device="cuda")
    if ctx.world > 1:
        import torch.distributed as dist
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms)


timed([1], False)                                   # warm-up: allocations, weight packing, NCCL channels
t_a = timed([2], False)
halo0 = tile.halo_bytes_moved
t_b = timed([6], False)                             # fixed costs (init, gather) cancel in the difference
ms_iter = (t_b - t_a) / 4
halo_iter = (tile.halo_bytes_moved - halo0) / 6
res = dict(ms_per_inference_iter=ms_iter)
if dm is not None:                                  # DDnet alone on this rank's strip, as the solver calls it
    eng = dm.engine()
    strip = torch.from_numpy(np.ascontiguousarray(np.moveaxis(sl(warm), 2, 0))).cuda()
    eng.forward_tiled(strip, tile)
    torch.cuda.synchronize(); ctx.barrier()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(3):
        eng.forward_tiled(strip, tile)
    e.record(); torch.cuda.synchronize()
    ms_dd = torch.tensor([s.elapsed_time(e) / 3], device="cuda")
    if ctx.world > 1:
        import torch.distributed as dist
        dist.all_reduce(ms_dd, op=dist.ReduceOp.MAX)
    res.update(ms_ddnet_per_iter=float(ms_dd), ddnet_share_of_iter=float(ms_dd) / ms_iter,
               ddnet_frame_chunk=eng.tiled_chunk_frames(B, tile))
if not a.no_update:
    t_u = timed([8, 2], True)                       # update at k = 9: 2 Adam steps + host noise for the whole frame
    res["ms_full_schedule_8_2_with_one_update"] = t_u
    res["ms_update_call_est"] = t_u - t_a - 8 * ms_iter
r = twoStageAdmm_denoise_bayer(*args[:5], [2], False, [12 / 255], **dict(kw, update_=False))   # quality / gather path once
if a.tv_warm_start:
    r_crude = twoStageAdmm_denoise_bayer(*args[:5], [2], False, [12 / 255], **dict(kw_crude, update_=False))
mem = torch.tensor([torch.cuda.max_memory_allocated() / 2**30], device="cuda")
mems = [mem.clone() for _ in range(ctx.world)]
halo = torch.tensor([halo_iter], device="cuda")
halos = [halo.clone() for _ in range(ctx.world)]
if ctx.world > 1:
    import torch.distributed as dist
    dist.all_gather(mems, mem)
    dist.all_gather(halos, halo)
if ctx.rank == 0:
    demosaic = "DDnet (synthetic weights)" if dm is not None else "Malvar"
    if a.close_form:
        demosaic += ", closed form from iteration 2"
    res.update({"config": "configs[4]: %dx%dx%d Bayer FastDVDnet, %s, %d row strips + halo exchange" % (H, W, B, demosaic,
                                                                                                        ctx.world),
                "n_gpus": ctx.world, "iters_per_sec": 1e3 / ms_iter, "psnr_2_iters": [round(float(p), 3) for p in r[4]],
                "halo_bytes_per_inference_iter_per_rank": [int(h) for h in halos],
                "peak_mem_GiB_per_rank": [round(float(v), 2) for v in mems]})
    if a.tv_warm_start:
        res.update({"warm_start": "tiled stage 1, 40 TV iterations", "ms_stage1_40_iters_first_call_rank0": ms_stage1,
                    "psnr_2_iters_crude_start": [round(float(p), 3) for p in r_crude[4]]})
    print(json.dumps(res))
ctx.finalize()
