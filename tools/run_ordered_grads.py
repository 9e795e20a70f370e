"""Cost of the fixed-order backward reductions on one GPU.

    python tools/run_ordered_grads.py --out DIR

* one FastDVDnet fine-tune call at 8 x 512 x 512 (two Adam steps, then the eval forward), CUDA events, median of 5;
* one online FastDVDnet reconstruction at 512 x 512 x 8 Bayer (iterations [21, 2], fine-tune every 3rd iteration), median of 3;
* in a separate torch.profiler run of one fine-tune call: kernel time per backward pass of the weight-gradient kernels, of the
  act_bwd / fused data-gradient kernels that produce column sums, and of the slot reductions (ordered_slot_sum_kernel).
The card's name and power limit are read in the same run.  Writes DIR/ordered_grads.json."""
import argparse
import io
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["nvidia_smi"] = q
    except (OSError, subprocess.SubprocessError):
        info["nvidia_smi"] = None
    return info


def timed(fn, n):
    ts = []
    for _ in range(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts)), ts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("run_ordered_grads.py measures on the GPU: no CUDA device")
    from adaptivepnp_sci_b200.dvp_linear_inv_2_stage_ADMM_tensor_online import np2tch_cuda, twoStageAdmm_denoise_bayer
    from adaptivepnp_sci_b200.fastdvdnet_adapter import DataParallelLike, finetune_and_denoise
    from adaptivepnp_sci_b200.fastdvdnet_models import FastDVDnet
    from adaptivepnp_sci_b200.synthetic import fastdvdnet_synthetic_state_dict, make_case
    from adaptivepnp_sci_b200.utilspy import worker_init_fn

    sd = {"module." + k: v for k, v in fastdvdnet_synthetic_state_dict().items()}

    def model():
        m = DataParallelLike(FastDVDnet())
        m.load_state_dict(sd)
        return m.eval().cuda()

    res = {"card": card()}
    meas, mask, orig = make_case(512, 512, 8, 3000, bayer=True)
    v = torch.from_numpy(orig).permute(2, 0, 1).unsqueeze(1).repeat(1, 3, 1, 1).contiguous().cuda()
    phi = torch.from_numpy(mask).permute(2, 0, 1).contiguous().cuda()
    y = torch.from_numpy(meas).cuda()
    m = model()
    np.random.seed(0)
    step = lambda: finetune_and_denoise(v, phi, y, 12 / 255, m, 2e-6, 2)
    step()                                                   # warm-up: plans, scratch buffers, the noise stream
    torch.cuda.synchronize()
    res["finetune_8x512x512_2steps_ms"], res["finetune_samples_ms"] = timed(step, 5)

    warm = np.clip(meas[:, :, None] * mask / np.maximum(mask.sum(2, keepdims=True), 1), 0, 1).astype(np.float32)

    def recon():
        worker_init_fn(0)
        twoStageAdmm_denoise_bayer(meas, mask, 1, 0.01, 'fastdvd_color', [21, 2], False, [12 / 255, 6 / 255],
                                   x0_bayer=np2tch_cuda(warm), X_orig=orig, model_denoise=m, show_iqa=False,
                                   demosaic_method='malvar2004', lr_=2e-6, interval_iter=3, logf=io.StringIO(), update_=True,
                                   update_per_iter=2, update_times=-1)
    recon()
    torch.cuda.synchronize()
    res["recon_512x512x8_fastdvd_online_ms"], res["recon_samples_ms"] = timed(recon, 3)

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    groups = {"wgrad": ("conv_wgrad2_tc_kernel", "conv_wgrad3_tc_kernel", "wgrad_ref_kernel"),
              "ordered_slot_sum": ("ordered_slot_sum_kernel",), "act_bwd": ("act_bwd_kernel",),
              "dgrad_fused_colsum": ("conv_fwd2_tc_kernel<1, 5", "conv_fwd2_tc_kernel<2, 5",
                                     "conv_fwd2_tc_kernel<1, 4", "conv_fwd2_tc_kernel<2, 4")}
    per = {k: {"us": 0.0, "launches": 0} for k in groups}
    for ev in prof.key_averages():
        for k, pats in groups.items():
            if any(p in ev.key for p in pats):
                per[k]["us"] += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
                per[k]["launches"] += ev.count
    backward_passes = 2
    res["per_backward"] = {k: {"kernel_ms": round(v["us"] / 1e3 / backward_passes, 4), "launches": v["launches"] // backward_passes}
                           for k, v in per.items()}
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "ordered_grads.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
