"""Stage 1 (TV warm start) of one large frame on row strips, against the un-tiled run.

    torchrun --nproc-per-node N tools/run_tiled_tv.py [--size 2048] [--frames 24] [--iters 40]

Every rank runs ``admm_denoise_bayer_demosaic_pre(..., tile=...)`` on its H/N rows of ``make_case(..., seed=5001)``.  Prints
one JSON line (rank 0):
  * ms per ADMM iteration (CUDA events, max over ranks; the difference of two run lengths, so set-up cancels);
  * the TV energies' all-gather, timed alone with CUDA events (same tensor, same process group) as ms per call and as a
    share of the iteration;
  * max |tiled - un-tiled| of the returned x, against an un-tiled run on rank 0's GPU (a 2048x2048x24 cube is 384 MiB),
    and the largest difference of the PSNR trajectories.  Given equal stop indices x is bit-identical; a stop index that
    differed in any of the TV calls would change every later iterate of that channel, so max-abs 0 also shows that the
    stops agreed."""
import argparse, json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from adaptivepnp_sci_b200 import parallel
from adaptivepnp_sci_b200.dvp_linear_inv_2_stage_ADMM_tensor_online import admm_denoise_bayer_demosaic_pre
from adaptivepnp_sci_b200.synthetic import make_case

ap = argparse.ArgumentParser()
ap.add_argument("--size", type=int, default=2048)
ap.add_argument("--frames", type=int, default=24)
ap.add_argument("--iters", type=int, default=40)
a = ap.parse_args()
ctx = parallel.init()
H = W = a.size
B = a.frames
tile = parallel.TileContext(ctx, H, W)
meas, mask, orig = make_case(H, W, B, 5001, bayer=True)
sl = tile.slice_rows


def max_over_ranks(v):
    t = torch.tensor([v], dtype=torch.float64, device="cuda")
    if ctx.world > 1:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t)


def timed(n):
    torch.cuda.synchronize(); ctx.barrier()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    admm_denoise_bayer_demosaic_pre(sl(meas), sl(mask), 1, 0.01, 'tv', [n], False, [0], tile=tile, return_device=True)
    e.record(); torch.cuda.synchronize()
    return max_over_ranks(s.elapsed_time(e))


timed(2)                                            # warm-up: allocations, P2P mapping, communicator set-up
t_a, t_b = timed(4), timed(4 + a.iters)
ms_iter = (t_b - t_a) / a.iters

ms_gather = 0.0
if ctx.world > 1:                                   # the all-gather of TileContext.tv_chambolle, alone
    import torch.distributed as dist
    esum = torch.zeros((4 * B, 8), dtype=torch.float64, device="cuda")
    out = torch.empty((ctx.world, 4 * B, 8), dtype=torch.float64, device="cuda")
    for _ in range(10):
        dist.all_gather_into_tensor(out, esum)
    torch.cuda.synchronize(); ctx.barrier()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(200):
        dist.all_gather_into_tensor(out, esum)
    e.record(); torch.cuda.synchronize()
    ms_gather = max_over_ranks(s.elapsed_time(e) / 200)

tiled = admm_denoise_bayer_demosaic_pre(sl(meas), sl(mask), 1, 0.01, 'tv', [a.iters], False, [0], X_orig=sl(orig),
                                        tile=tile)
used_p2p = tile.p2p is not None
if tile.p2p is not None:
    tile.p2p.close()
if ctx.rank == 0:
    ref = admm_denoise_bayer_demosaic_pre(meas, mask, 1, 0.01, 'tv', [a.iters], False, [0], X_orig=orig)
    dev = torch.cuda.get_device_properties(0)
    try:                                            # the power limit is part of the number
        import subprocess
        plim = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        plim = "unknown"
    res = {"config": "stage 1 TV, %dx%dx%d Bayer, %d row strips" % (H, W, B, ctx.world), "n_gpus": ctx.world,
           "gpu": dev.name, "power_limit": plim, "iters": a.iters, "ms_per_iter": round(ms_iter, 4),
           "ms_all_gather_alone": round(ms_gather, 4), "all_gather_share": round(ms_gather / ms_iter, 4),
           "max_abs_x_vs_untiled": float(np.max(np.abs(tiled[0] - ref[0]))),
           "max_abs_psnr_trajectory_dB": float(np.max(np.abs(np.array(tiled[3]) - np.array(ref[3])))),
           "psnr_final_dB": round(float(ref[3][-1]), 4), "halo_peer_to_peer": used_p2p}
    print(json.dumps(res))
ctx.finalize()
