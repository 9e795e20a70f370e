"""Grayscale video SCI with online FastDVDnet ('fastdvd_gray') at the standard 256x256x8 case: timing of whole
reconstructions, with and without the online update, and the CPU time of the derived oracle.

    python tools/run_gray_fastdvd.py --out DIR        -> DIR/gray_fastdvd.json

Input make_case(256, 256, 8, seed=1001, bayer=False); warm start: 40 TV iterations (stage 1); then the FastDVDnet script
schedule: sigma [12, 6]/255, iterations [21, 2], an update every 9 iterations (k = 9, 18) of 2 Adam steps at lr 2e-6,
synthetic gray weights.  Every reconstruction starts from the same weights and the same numpy RNG state.  CUDA events around
whole reconstructions: 3 warm-ups, the median of 10.  FLOPs are the algorithmic ones of one inference pass (both DenBlocks,
B centre frames each), counted from the gray model's layer shapes."""
import argparse
import io
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

H, W, B = 256, 256, 8
SCHED = dict(iter_max=[21, 2], sigma=[12 / 255, 6 / 255], lr_=2e-6, interval_iter=9, update_per_iter=2)


def inference_flops(net, B, H, W):
    """2 * MACs of the 16 convolutions of both DenBlocks of ``net`` (gray shapes), B triples per block."""
    total = 0
    for blk in (net.temp1, net.temp2):
        h, w = H, W
        for conv, _, _, stride, ps in blk.conv_specs():
            ho, wo = (h - 1) // stride + 1, (w - 1) // stride + 1
            total += 2 * B * ho * wo * 9 * (conv.in_channels // conv.groups) * conv.out_channels
            h, w = (2 * ho, 2 * wo) if ps else (ho, wo)
    return total


def card():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit",
                        "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().split(", ") + [None, None])[:2] if q.returncode == 0 else (None, None)
    return {"name": name or torch.cuda.get_device_name(), "power_limit": power}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("run_gray_fastdvd.py measures on the GPU: no CUDA device")
    from adaptivepnp_sci_b200.dvp_linear_inv_2_stage_ADMM_tensor_online import (admm_denoise_bayer_demosaic_pre,
                                                                                twoStageAdmm_denoise_gray)
    from adaptivepnp_sci_b200.fastdvdnet_adapter import DataParallelLike
    from adaptivepnp_sci_b200.fastdvdnet_models import FastDVDnet
    from adaptivepnp_sci_b200.synthetic import fastdvdnet_gray_synthetic_state_dict, make_case
    from oracle import gray_fastdvd, networks

    meas, mask, orig = make_case(H, W, B, 1001, bayer=False)
    warm = admm_denoise_bayer_demosaic_pre(meas, mask, 1, 0.01, 'tv', [40], False, [0], X_orig=orig, show_iqa=False)[0]
    sd = {"module." + k: v for k, v in fastdvdnet_gray_synthetic_state_dict().items()}
    model = DataParallelLike(FastDVDnet(num_input_frames=5, num_color_channels=1)).eval().cuda()
    x0 = torch.from_numpy(np.ascontiguousarray(warm)).cuda()

    def run(update):
        model.load_state_dict(sd, strict=True)
        model.module.engine()                                    # the twin takes the weights outside the timed region
        np.random.seed(0)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = twoStageAdmm_denoise_gray(meas, mask, 'fastdvd_gray', x0=x0, X_orig=orig, model_denoise=model,
                                      logf=io.StringIO(), update_=update, **SCHED)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), r

    n_iter = sum(SCHED["iter_max"])
    res = {"case": "make_case(%d, %d, %d, seed=1001, bayer=False), warm start 40 TV iterations" % (H, W, B),
           "schedule": SCHED, "admm_iterations": n_iter, "card": card()}
    for update in (True, False):
        for _ in range(3):
            run(update)
        times, r = [], None
        for _ in range(10):
            t, r = run(update)
            times.append(t)
        ms = float(np.median(times))
        res["update" if update else "no_update"] = {
            "ms_per_reconstruction": ms, "admm_it_per_s": n_iter / (ms / 1e3), "ms_all": times,
            "psnr_mean_db": float(np.mean(r[2])), "psnr_last_iteration_db": float(r[4][-1])}
    u, n = res["update"]["ms_per_reconstruction"], res["no_update"]["ms_per_reconstruction"]
    res["update_share_of_reconstruction"] = (u - n) / u
    res["inference_pass_flops"] = inference_flops(model.module, B, H, W)
    res["inference_pass_flops_note"] = "algorithmic, gray layer shapes, %dx%dx%d, both DenBlocks" % (H, W, B)
    # the derived oracle (CPU PyTorch), 2 iterations of the same loop (no update falls in them)
    om = networks.Wrapped(networks.FastDVDnet(5, 1))
    om.load_state_dict(sd, strict=True)
    t0 = time.perf_counter()
    gray_fastdvd.twoStageAdmm_denoise_gray(meas, mask, 'fastdvd_gray', iter_max=[2], sigma=[12 / 255],
                                           x0=torch.from_numpy(warm), X_orig=orig, model_denoise=om.eval(), lr_=2e-6,
                                           interval_iter=9, update_=True, update_per_iter=2)
    res["oracle_cpu_s_2_iterations"] = time.perf_counter() - t0
    res["oracle_cpu_threads"] = torch.get_num_threads()
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "gray_fastdvd.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k not in ("schedule",)}, default=str)[:2000])
    print("wrote", path)


if __name__ == "__main__":
    main()
