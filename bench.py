#!/usr/bin/env python
"""Benchmark of the AdaptivePnP_SCI hot path on B200 - headline: two-stage online-adaptive ADMM reconstruction,
512x512x8 Bayer, FastDVDnet (BASELINE.json configs[3]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 1..5] [--dump-outputs DIR]

Contract (see the task statement): W untimed warm-up steps, exactly K timed steps bracketed by a barrier +
torch.cuda.synchronize() on both sides, CUDA-event timing, max over ranks, rank 0 prints ONE JSON line.

--config selects the BASELINE.json configuration (1-based; the default 4 is the one the metric is quoted on):
  1  ADMM-TV warm start, 256x256x8 gray cube, 40 iterations            (replicas: one cube per GPU, weak)
  2  two-stage ADMM + online FFDNet-gray, 256x256x8 (derived loop)     (replicas, weak)
  3  512x512x8 Bayer, FFDNet-colour + Malvar, iterations 6/6/4         (one measurement group per GPU, own weights, weak)
  4  512x512x8 Bayer, online FastDVDnet, iterations 21/2               (one group per GPU, shared weights: NCCL grad all-reduce, weak)
  5  2048x2048x24 Bayer, FastDVDnet, iterations 8/2, inference         (ONE frame, row strips + halo exchange, strong)
One STEP is one full reconstruction of the configuration's unit.  metric = ADMM iterations / second (whole job);
`sec_per_recon` is reported beside it.

* value   = inputs resident in HBM, outputs left on the device.
* e2e     = the public drop-in call (numpy in, numpy out): H2D of y, Phi and the warm start and D2H of the
            reconstructions inside the timed region (pinned host buffers).
* roofline       = the dominant kernel of the configuration (conv for the deep denoisers, TV for config 1).
* roofline_hbm   = event-timed GB/s of the HBM-bound kernels (projection, Malvar, dual update, TV) at the
                   configuration's cube size, L2 flushed between launches.
* cpu_baseline   = the oracle's CPU restatement of the reference (== the reference bit for bit, tests/golden/make_golden.py)
                   on the host cores, a bounded sample extrapolated to the schedule (the sample is described).
* gpu_eager_baseline = the UNMODIFIED reference (baseline/_ref, copied by baseline/install_ref.py) on the same B200
                   through PyTorch eager: the honest same-box comparator.  null when baseline/_ref is absent.
* delta_psnr     = configs 3/4, N = 1: the reconstruction against what the REFERENCE produced for the same inputs
                   (tests/golden/fullsize.npz, generated on the CPU by tests/golden/make_golden_fullsize.py).
* --impl reference = the oracle port on the host cores (the reference is pure Python and cannot be pip-installed);
                   each step a bounded sample, the fine-tune iteration timed once and mixed in per the real schedule.
"""
import argparse
import io
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LR, UPDATE_PER_ITER = 2e-6, 2
CFG = {
    1: dict(H=256, W=256, B=8, bayer=False, seed=1001, iters=[40], sigma=[0], denoiser="tv", interval=None, scaling="weak",
            workload="configs[0]: ADMM-TV warm start, 256x256x8 gray cube, 40 iterations, one cube per GPU per step"),
    2: dict(H=256, W=256, B=8, bayer=False, seed=1001, iters=[6, 6, 4], sigma=[25 / 255, 12 / 255, 6 / 255], denoiser="ffdnet_gray",
            interval=6, scaling="weak",
            workload="configs[1]: two-stage ADMM + online FFDNet-gray, 256x256x8 (derived loop, SURVEY 8(c)), one cube per GPU per step"),
    3: dict(H=512, W=512, B=8, bayer=True, seed=3000, iters=[6, 6, 4], sigma=[25 / 255, 12 / 255, 6 / 255], denoiser="ffdnet_color",
            interval=6, scaling="weak",
            workload="configs[2]: 512x512x8 Bayer, FFDNet-colour + Malvar, online update, 1 measurement group per GPU per step (own weights)"),
    4: dict(H=512, W=512, B=8, bayer=True, seed=3000, iters=[21, 2], sigma=[12 / 255, 6 / 255], denoiser="fastdvd_color",
            interval=9, scaling="weak",
            workload="configs[3]: two-stage ADMM + online FastDVDnet, 512x512x8 Bayer, 1 measurement group per GPU per step"),
    5: dict(H=2048, W=2048, B=24, bayer=True, seed=5001, iters=[8, 2], sigma=[12 / 255, 6 / 255], denoiser="fastdvd_color",
            interval=9, scaling="strong",
            workload="configs[4]: 2048x2048x24 Bayer, FastDVDnet, iterations 8/2 (inference), ONE frame in row strips over the GPUs + halo exchange"),
}


def config_dict(c, cfg):
    d = {"workload": cfg["workload"], "baseline_config": c, "iters_per_recon": int(sum(cfg["iters"])),
         "sigma_x255": [round(s * 255) for s in cfg["sigma"]], "iter_max": cfg["iters"],
         "l2": "working set per step >> 126 MB L2 (solver state + activations): no flush needed; roofline_hbm flushes L2 between launches"}
    if cfg["denoiser"] == "fastdvd_color":
        d["weights"] = "synthetic contractive init seed 4242 (trained FastDVDnet weights absent from the reference)"
        d["conv"] = "tcgen05: inference passes kind::f16 (fp16 operands, same 11-bit significand as TF32), online update kind::tf32; fp32 accumulate"
        d["finetune"] = "k=9,18; 2 Adam steps; lr 2e-6" if c == 4 else "none (inference schedule; the fine-tune of one 2048x2048x24 frame needs all 8 GPUs)"
    elif cfg["denoiser"].startswith("ffdnet"):
        d["weights"] = "model_zoo/%s.pth (the reference's own file)" % cfg["denoiser"]
        d["conv"] = ("tcgen05: inference passes kind::f16 with every weight and activation as fp16 value + fp16 remainder x 2^11 "
                     "(3 products, two fp32 accumulators: ~fp32 accuracy); online update kind::tf32 with split weights")
        d["finetune"] = "k=6,12; 2 Adam steps; lr 2e-6"
    return d


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.t.join(timeout=2)
        sm = sorted(float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit())
        reasons = set()
        for r in self.rows:
            if len(r) >= 7:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        out = {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
               "reasons": sorted(reasons), "samples": len(sm)}
        if getattr(self, "extended", False):
            out["note"] = "timed region < 1 s: the same step kept running (untimed) under the sampler for 1 s more"
        return out


# ---------------------------------------------------------------------------------------------------------------------
# reference legs: the oracle port on the host cores (cpu_baseline / --impl reference) and the unmodified reference on
# the GPU through PyTorch eager (gpu_eager_baseline).  The only parts of this file that touch oracle/.
# ---------------------------------------------------------------------------------------------------------------------
def _crude_warm(meas, mask):
    return np.clip(meas[:, :, None] * mask / np.maximum(mask.sum(2, keepdims=True), 1), 0, 1).astype(np.float32)


def _oracle_models(cfg):
    from oracle import networks, synthetic
    if cfg["denoiser"] == "fastdvd_color":
        m = networks.Wrapped(networks.FastDVDnet())
        m.load_state_dict({"module." + k: v for k, v in synthetic.fastdvdnet_synthetic_state_dict().items()}, strict=True)
    elif cfg["denoiser"] == "ffdnet_color":
        m = networks.FFDNet(3, 3, 96, 12, 'R')
        m.load_state_dict(torch.load(os.path.join(ROOT, "model_zoo", "ffdnet_color.pth")), strict=True)
    else:
        m = networks.FFDNet(1, 1, 64, 15, 'R')
        m.load_state_dict(torch.load(os.path.join(ROOT, "model_zoo", "ffdnet_gray.pth")), strict=True)
    return m.eval()


class CpuReference:
    """Bounded samples of the configuration's schedule on the host cores, oracle port of the reference."""

    def __init__(self, c):
        from oracle import synthetic
        torch.set_num_threads(os.cpu_count() or 1)
        self.c, self.cfg = c, CFG[c]
        cfg = self.cfg
        self.rows = cfg["H"]
        self.scale = 1.0
        if c == 5:
            # one inference iteration of the whole 2048x2048x24 frame is minutes of CPU time: the sample is a 256-row strip
            # (1/8 of the pixels; per-pixel work is uniform), scaled by 8
            self.rows, self.scale = 256, cfg["H"] / 256.0
        meas, mask, orig = synthetic.make_case(self.rows, cfg["W"], cfg["B"], cfg["seed"], bayer=cfg["bayer"])
        self.meas, self.mask, self.orig = meas, mask, orig
        self.warm = _crude_warm(meas, mask)
        self.t_ft = None
        self.cores = torch.get_num_threads()

    def _run(self, iters, update, interval=None):
        from oracle import admm
        cfg = self.cfg
        t0 = time.perf_counter()
        if cfg["denoiser"] == "tv":
            admm.admm_denoise_bayer_demosaic_pre(self.meas, self.mask, 1, 0.01, 'tv', iters, False, [0], x0_bayer=None,
                                                 X_orig=None, show_iqa=False)
        elif cfg["denoiser"] == "ffdnet_gray":
            admm.twoStageAdmm_denoise_gray(self.meas, self.mask, 'ffdnet_gray', iter_max=iters, sigma=[cfg["sigma"][0]],
                                           x0=torch.from_numpy(self.warm), X_orig=None, model_denoise=_oracle_models(cfg),
                                           show_iqa=False, lr_=LR, interval_iter=interval or cfg["interval"], update_=update,
                                           update_per_iter=UPDATE_PER_ITER)
        else:
            kw = dict(update_times=-1) if cfg["denoiser"] == "fastdvd_color" else {}
            admm.twoStageAdmm_denoise_bayer(self.meas, self.mask, 1, 0.01, cfg["denoiser"], iters, False, [cfg["sigma"][0]],
                                            x0_bayer=torch.from_numpy(self.warm), X_orig=None, model_denoise=_oracle_models(cfg),
                                            show_iqa=False, lr_=LR, interval_iter=interval or cfg["interval"], update_=update,
                                            update_per_iter=UPDATE_PER_ITER, **kw)
        return time.perf_counter() - t0

    def inference_iter(self):
        """seconds per inference ADMM iteration of the full-size unit."""
        n = 40 if self.c == 1 else 1
        return self._run([n], False) / n * self.scale

    def finetune_iter(self, t_inf):
        """seconds of ONE iteration with the online update (2 Adam steps + the final denoise), timed once and cached:
        3 iterations with the update at k = 2 (interval 2) minus two inference iterations."""
        if self.t_ft is None:
            self.t_ft = max(self._run([3], True, interval=2) * self.scale - 2 * t_inf, t_inf)
        return self.t_ft

    def n_updates(self):
        cfg = self.cfg
        if cfg["interval"] is None or self.c == 5:
            return 0
        return sum(1 for k in range(int(sum(cfg["iters"]))) if k > 1 and k % cfg["interval"] == 0)

    def schedule_seconds(self, t_inf):
        n, nu = int(sum(self.cfg["iters"])), self.n_updates()
        t = (n - nu) * t_inf
        if nu:
            t += nu * self.finetune_iter(t_inf)
        return t

    def describe(self):
        nu = self.n_updates()
        s = "oracle port of the reference loop on %d host threads: " % self.cores
        if self.c == 1:
            return s + "the full 40-iteration reconstruction"
        s += "1 inference ADMM iteration timed per sample"
        if self.c == 5:
            s += " on a 256-row strip of the frame (x8)"
        if nu:
            s += "; the iteration with the online update (2 Adam steps + final denoise, full size) timed once (%.1f s) and " \
                 "mixed in per the schedule (%d of %d iterations)" % (self.t_ft or -1, nu, int(sum(self.cfg["iters"])))
        return s


def run_reference(args):
    """--impl reference: CPU port of the reference loop, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    c = args.config
    cfg = CFG[c]
    ref = CpuReference(c)
    n = int(sum(cfg["iters"]))
    for _ in range(args.warmup):
        ref.inference_iter()
    t = 0.0
    for _ in range(args.steps):
        t += ref.schedule_seconds(ref.inference_iter())
    v = args.steps * n / t
    _emit({"impl": "reference", "metric": "admm_iters_per_sec", "value": v, "unit": "iters/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "sec_per_recon": t / args.steps,
           "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": config_dict(c, cfg),
           "cpu_baseline": {"value": v, "unit": "iters/s", "cores": ref.cores, "kind": "port", "sample": ref.describe()},
           "e2e": {"value": v, "unit": "iters/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})


def gpu_eager_baseline(c, cfg, meas, mask, orig, warm):
    """The UNMODIFIED reference (baseline/_ref) on this GPU through PyTorch eager, same inputs, same schedule."""
    from oracle import ref_harness
    if c == 2:
        return {"value": None, "why": "the reference has no function for the gray two-stage loop (SURVEY 8(c))"}
    if not ref_harness.available(ref_harness.BASELINE_REF):
        return {"value": None, "why": "baseline/_ref absent (run baseline/install_ref.py in the build container)"}
    try:
        ns = ref_harness.load(root=ref_harness.BASELINE_REF, device="cuda")
        from oracle import synthetic
        n = int(sum(cfg["iters"]))

        def model():
            if cfg["denoiser"] == "fastdvd_color":
                m = torch.nn.DataParallel(ns.fastdvd_models.FastDVDnet(num_input_frames=5), device_ids=[torch.cuda.current_device()])
                m.load_state_dict({"module." + k: v for k, v in synthetic.fastdvdnet_synthetic_state_dict().items()}, strict=True)
                return m.eval().cuda()
            if cfg["denoiser"] == "ffdnet_color":
                m = ns.network_ffdnet.FFDNet(in_nc=3, out_nc=3, nc=96, nb=12, act_mode='R')
                m.load_state_dict(torch.load(os.path.join(ROOT, "model_zoo", "ffdnet_color.pth")), strict=True)
                return m.eval().cuda()
            return None

        def run(iters, sigma, update):
            ns.utilspy.worker_init_fn(0)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            with contextlib_redirect():
                if cfg["denoiser"] == "tv":
                    ns.dvp.admm_denoise_bayer_demosaic_pre(meas, mask, 1, 0.01, 'tv', iters, False, [0], x0_bayer=None, X_orig=None,
                                                           model=None, show_iqa=False, logf=io.StringIO())
                else:
                    kw = dict(update_times=-1) if cfg["denoiser"] == "fastdvd_color" else {}
                    ns.dvp.twoStageAdmm_denoise_bayer(meas, mask, 1, 0.01, cfg["denoiser"], iters, False, sigma,
                                                      x0_bayer=torch.from_numpy(warm).cuda(), X_orig=None, model_denoise=model(),
                                                      model_demosaic=None, show_iqa=False, demosaic_method='malvar2004', lr_=LR,
                                                      interval_iter=cfg["interval"], logf=io.StringIO(), update_=update,
                                                      update_per_iter=UPDATE_PER_ITER, **kw)
            torch.cuda.synchronize()
            return time.perf_counter() - t0
        out = {"unit": "iters/s", "what": "unmodified reference (baseline/_ref), PyTorch %s eager on the same GPU, numpy in / numpy out; "
               "TV / PSNR come from the restated scikit-image routines (absent in the image)" % torch.__version__}
        if c == 5:
            iters, sigma, update, n_run = [2], [cfg["sigma"][0]], False, 2
            out["sample"] = "2 inference iterations of the full 2048x2048x24 frame on ONE GPU (the reference has no multi-GPU path)"
        else:
            iters, sigma, update, n_run = cfg["iters"], cfg["sigma"], c in (3, 4), n
            out["sample"] = "the full schedule (incl. the online updates)" if update else "the full schedule"
        for name, tf32 in (("fp32", False), ("default", True)):
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cuda.matmul.allow_tf32 = False
            run([2] if c != 1 else [2], sigma[:1], False)                 # warm-up: cuDNN heuristics, allocator
            t = run(iters, sigma, update)
            key = "" if name == "fp32" else "_cudnn_tf32_allowed"
            out["value" + key] = n_run / t
            out["sec_per_recon" + key] = t * (n / n_run)
        out["precision"] = "value: fp32 convolutions (torch.backends.cudnn.allow_tf32=False); value_cudnn_tf32_allowed: PyTorch's default"
        torch.backends.cudnn.allow_tf32 = True
        torch.cuda.empty_cache()
        return out
    except Exception as e:                                                 # a baseline failure must not lose the bench line
        return {"value": None, "why": "%s: %s" % (type(e).__name__, str(e)[:200])}


class contextlib_redirect:
    """Silence the reference's print() calls (loss lines, tqdm) without touching the real stdout of the JSON line."""

    def __enter__(self):
        self._o = sys.stdout
        sys.stdout = io.StringIO()

    def __exit__(self, *a):
        sys.stdout = self._o


# ---------------------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------------------
def hbm_kernel_table(H, W, B, dev, pk):
    """Event-timed algorithmic GB/s of the HBM-bound kernels at this cube size (SURVEY 8(d) byte counts), L2 flushed."""
    from adaptivepnp_sci_b200 import ops
    cube, plane = H * W * B * 4, H * W * 4
    g = torch.Generator(device=dev).manual_seed(0)
    theta = torch.rand(B, H, W, device=dev, generator=g)
    b = 0.1 * torch.randn(B, H, W, device=dev, generator=g)
    phi = (torch.rand(B, H, W, device=dev, generator=g) > 0.5).float()
    y = (theta * phi).sum(0)
    phisum = phi.sum(0).clamp_(min=1)
    x, b2 = torch.empty_like(theta), torch.empty_like(b)
    w = torch.randn(B, 3, H, W, device=dev, generator=g)
    x_rgb, u = torch.empty_like(w), torch.empty_like(w)
    xhat = torch.rand(B, 3, H, W, device=dev, generator=g)
    ws = ops.TvWorkspace(H, W, B, dev)
    flush = torch.zeros(64 * 1024 * 1024, device=dev)                     # 256 MB > 126 MB L2
    cases = [("project_stage1", lambda: ops.project_stage1(theta, b, phi, y, phisum, x, 1.0, 0.01), 4 * cube + 2 * plane),
             ("project_stage2", lambda: ops.project_stage2(theta, b, phi, y, phisum, x, 1.0, 0.55), 4 * cube + 2 * plane),
             ("tv_chambolle(+clip+dual)", lambda: ops.tv_chambolle(x, b, -1.0, theta, b2, -1.0, True, ws), 4 * cube),
             ("malvar2004(+w/tau)", lambda: ops.malvar2004(x, b, 1.0, w, 0.01, x_rgb, u), 11 * cube),
             ("dual_update_rgb", lambda: ops.dual_update_rgb(xhat, x_rgb, w, x, b, theta, False), 13 * cube)]
    rows = []
    for name, fn, nbytes in cases:
        for _ in range(3):
            fn()
        ts = []
        for _ in range(9):
            flush.add_(1.0)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record(); fn(); e.record()
            torch.cuda.synchronize()
            ts.append(s.elapsed_time(e) * 1e-3)
        t = sorted(ts)[len(ts) // 2]
        rows.append({"kernel": name, "bytes": nbytes, "ms": 1e3 * t, "achieved": nbytes / t / 1e9, "frac": nbytes / t / 1e9 / pk})
    return rows


# what the timed call returns, in order, per configuration (non-array members of the returned tuple are not named):
# config 1 the stage-1 Bayer cube [H,W,B]; config 2 the gray denoiser output and theta [H,W,B]; configs 3-5 the planar device
# tensors xhat [B,3,H,W] and theta [B,H,W] (config 5: rank 0's row strip)
OUTPUT_NAMES = {1: ("x_bayer",), 2: ("xhat", "theta"), 3: ("xhat", "theta"), 4: ("xhat", "theta"), 5: ("xhat", "theta")}
DUMP_LIMIT_BYTES = 63 * 1024 * 1024          # array data; the .npy headers stay well inside the last of 64 MB


def dump_outputs(d, names, out):
    """DIR/<name>.npy of every named output of one step.  Above 63 MB of data in all, every array is replaced by the same
    fixed strided sample of its flattened elements (every s-th, s = ceil(total / 63 MB)), so two runs stay comparable."""
    arrays = []
    for name, a in zip(names, out):
        if isinstance(a, np.ndarray):
            a = torch.from_numpy(a)
        arrays.append((name, a.detach()))
    total = sum(a.numel() * (8 if a.dtype == torch.float64 else 4) for _, a in arrays)
    stride = -(-total // DUMP_LIMIT_BYTES)
    os.makedirs(d, exist_ok=True)
    for name, a in arrays:
        if a.dtype != torch.float64:
            a = a.float()
        a = a.contiguous()
        if stride > 1:
            a = a.view(-1)[::stride]
        np.save(os.path.join(d, name + ".npy"), a.cpu().numpy())
        sys.stderr.write("bench: %s/%s.npy %s%s\n" % (d, name, tuple(a.shape),
                                                         " (every %d-th element)" % stride if stride > 1 else ""))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=4, choices=[1, 2, 3, 4, 5])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-eager", action="store_true")
    ap.add_argument("--no-delta-psnr", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (rank 0) as DIR/<name>.npy, for output-by-output comparison "
                         "of two builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)
    c = args.config
    cfg = CFG[c]
    H, W, B = cfg["H"], cfg["W"], cfg["B"]
    n_iter = int(sum(cfg["iters"]))

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    from adaptivepnp_sci_b200 import _lib, parallel
    from adaptivepnp_sci_b200.dvp_linear_inv_2_stage_ADMM_tensor_online import (admm_denoise_bayer_demosaic_pre,
                                                                                twoStageAdmm_denoise_bayer,
                                                                                twoStageAdmm_denoise_gray)
    from adaptivepnp_sci_b200.fastdvdnet_adapter import DataParallelLike
    from adaptivepnp_sci_b200.fastdvdnet_models import FastDVDnet
    from adaptivepnp_sci_b200.network_ffdnet import FFDNet
    from adaptivepnp_sci_b200.synthetic import fastdvdnet_synthetic_state_dict, make_case
    from adaptivepnp_sci_b200.utilspy import worker_init_fn

    # ---- setup (untimed): data of this rank's unit, warm start (stage 1, our kernels), model
    tile = None
    if c == 5:
        ctx = parallel.Context(rank, world, local_rank, "nccl")
        tile = parallel.TileContext(ctx, H, W)
        meas_f, mask_f, orig_f = make_case(H, W, B, cfg["seed"], bayer=True)
        warm_f = _crude_warm(meas_f, mask_f)                               # the TV stage does not tile; a crude At-normalised start
        meas, mask, orig, warm = (tile.slice_rows(a) for a in (meas_f, mask_f, orig_f, warm_f))
    else:
        meas, mask, orig = make_case(H, W, B, cfg["seed"] + rank, bayer=cfg["bayer"])
        warm = None
        if c != 1:
            warm = admm_denoise_bayer_demosaic_pre(meas, mask, 1, 0.01, 'tv', [40], False, [0], x0_bayer=None, X_orig=None,
                                                   show_iqa=False)[0]
    model, sd0 = None, None
    if cfg["denoiser"] == "fastdvd_color":
        sd0 = {"module." + k: v for k, v in fastdvdnet_synthetic_state_dict().items()}
        model = DataParallelLike(FastDVDnet(num_input_frames=5))
    elif cfg["denoiser"] == "ffdnet_color":
        sd0 = torch.load(os.path.join(ROOT, "model_zoo", "ffdnet_color.pth"))
        model = FFDNet(3, 3, 96, 12, 'R')
    elif cfg["denoiser"] == "ffdnet_gray":
        sd0 = torch.load(os.path.join(ROOT, "model_zoo", "ffdnet_gray.pth"))
        model = FFDNet(1, 1, 64, 15, 'R')
    if model is not None:
        model.load_state_dict(sd0, strict=True)
        model = model.eval().cuda()
    w0 = None

    def engine():
        return model.module.engine() if hasattr(model, "module") else model.engine()

    def grad_sync(g):
        if world > 1:
            dist.all_reduce(g, op=dist.ReduceOp.AVG)

    def reset_model():
        nonlocal w0
        if model is None or c == 5:
            return
        eng = engine()
        eng.prepare(False)
        if w0 is None:
            w0 = eng.bucket.flat.clone()
        else:
            eng.bucket.flat.copy_(w0)
            eng.after_step()

    def pinned(a):
        t = torch.empty(a.shape, dtype=torch.float32, pin_memory=True)
        t.copy_(torch.from_numpy(np.ascontiguousarray(a)))
        return t
    p_meas, p_mask = pinned(meas), pinned(mask)
    p_warm = pinned(warm) if warm is not None else None
    d_meas, d_mask = p_meas.to(dev), p_mask.to(dev)
    d_warm = p_warm.to(dev) if warm is not None else None
    worker_init_fn(0)      # seeds = 42 once, like the reference scripts (the fine-tune noise stream then continues)

    def run(y, phi, x0, device_out):
        reset_model()
        if c == 1:
            return admm_denoise_bayer_demosaic_pre(y, phi, 1, 0.01, 'tv', cfg["iters"], False, [0], x0_bayer=None, X_orig=None,
                                                   show_iqa=False)
        if c == 2:
            return twoStageAdmm_denoise_gray(y, phi, 'ffdnet_gray', iter_max=cfg["iters"], sigma=cfg["sigma"], x0=x0, X_orig=None,
                                             model_denoise=model, show_iqa=False, lr_=LR, interval_iter=cfg["interval"],
                                             update_=True, update_per_iter=UPDATE_PER_ITER)
        kw = dict(model_denoise=model, model_demosaic=None, demosaic_method='malvar2004', lr_=LR, interval_iter=cfg["interval"],
                  update_=(c in (3, 4)), update_per_iter=UPDATE_PER_ITER)
        if cfg["denoiser"] == "fastdvd_color":
            kw["update_times"] = -1
        if c == 4:
            kw["grad_sync"] = grad_sync                                   # shared weights: NCCL mean all-reduce of the gradients
        if c == 5:
            kw["tile"] = tile
        if device_out:
            kw["return_device"] = True                                   # config 5: the rank's own strips stay on its GPU
        return twoStageAdmm_denoise_bayer(y, phi, 1, 0.01, cfg["denoiser"], cfg["iters"], False, cfg["sigma"], x0_bayer=x0,
                                          X_orig=None, show_iqa=False, logf=None, **kw)

    def step_device():
        return run(d_meas, d_mask, d_warm, True)

    def step_e2e():
        # inputs start in PINNED host memory and go through the public call, results come back as host arrays (config 5:
        # every rank uploads its own strip; rank 0 alone assembles the full-frame result and copies it to the host)
        if tile is not None:
            tile.gather_root_only = True
        return run(p_meas.numpy(), p_mask.numpy(), p_warm.to(dev, non_blocking=True) if p_warm is not None else None, False)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = _lib.launch_count
        s.record()
        out = None
        for _ in range(steps):
            out = None      # a job drops (writes out) the previous result before the next reconstruction: its page-locked
            out = fn()      # buffers go back to the allocator instead of forcing a fresh cudaHostAlloc (1 s for 1.6 GB)
        e.record()
        barrier()
        ms = s.elapsed_time(e)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms, _lib.launch_count - l0, out

    units = 1 if c == 5 else world                                         # config 5: all ranks work on ONE frame
    for _ in range(args.warmup):
        step_device()
    clocks = ClockSampler(local_rank) if rank == 0 else None
    ms, launches, out = timed(step_device, args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, OUTPUT_NAMES[c], out)
    if clocks is not None and world == 1 and ms < 1000.0:
        # a timed region shorter than nvidia-smi's start-up (config 1: a few ms per step) would end without a sample: keep the
        # SAME step running under the sampler for about a second more (untimed) so that the line still carries clocks under load
        t_end = time.time() + 1.0
        while time.time() < t_end:
            step_device()
        torch.cuda.synchronize()
        clocks.extended = True
    clk = clocks.stop() if clocks else None
    value = units * args.steps * n_iter / (ms * 1e-3)
    for _ in range(2):          # untimed: page-locked staging buffers, allocator pools and the noise helper reach steady state
        step_e2e()
    ms_e2e, _, out_e2e = timed(step_e2e, args.steps)
    e2e_value = units * args.steps * n_iter / (ms_e2e * 1e-3)
    n_upd = sum(1 for k in range(n_iter) if c == 4 and k > 1 and k % cfg["interval"] == 0)
    h2d = p_meas.numel() * 4 + p_mask.numel() * 4 + (p_warm.numel() * 4 if p_warm is not None else 0) + n_upd * B * 3 * H * W * 8
    res = [a for a in out_e2e if isinstance(a, np.ndarray)]
    d2h = int(sum(a.nbytes for a in res))

    if rank != 0:
        if world > 1:
            # ranks > 0 of the tiled config take part in rank 0's extra tiled passes below? no: those run un-tiled on rank 0
            dist.destroy_process_group()
        return
    pk, pk_kind = peaks()
    # ---- roofline of the dominant kernel
    roofline = None
    if cfg["denoiser"] in ("fastdvd_color", "ffdnet_color", "ffdnet_gray"):
        eng = engine()
        hh = 512 if c == 5 else H                                          # per-layer profile of config 5 on a 512-row strip
        bb = 8 if c == 5 else B
        ch = 1 if cfg["denoiser"] == "ffdnet_gray" else 3
        u = torch.rand(bb, ch, hh, W, device=dev)
        eng.forward(u, cfg["sigma"][0])
        eng.profile = []
        eng.forward(u, cfg["sigma"][0])
        torch.cuda.synchronize()
        prof, eng.profile = eng.profile, None
        if os.environ.get("SCI_BENCH_VERBOSE"):
            for ev0, ev1, fl, tag in prof:
                t_ms = ev0.elapsed_time(ev1)
                sys.stderr.write("  %-28s %8.3f ms %8.1f TFLOP/s\n" % (tag, t_ms, fl / t_ms / 1e9))
        flops = sum(p[2] for p in prof)
        conv_s_serial = sum(p[0].elapsed_time(p[1]) for p in prof) * 1e-3   # an event pair per launch: serialises the chain
        # the chain as the solver runs it (launches back to back, programmatic dependent launch): CUDA events around whole passes;
        # the pass also contains its two small boundary kernels (input packing / output unpacking), which makes this conservative
        for _ in range(3):
            eng.forward(u, cfg["sigma"][0])
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n_pass = 10
        ev0.record()
        for _ in range(n_pass):
            eng.forward(u, cfg["sigma"][0])
        ev1.record()
        torch.cuda.synchronize()
        conv_s = ev0.elapsed_time(ev1) * 1e-3 / n_pass
        achieved = flops / conv_s / 1e12
        peak_bf16 = pk["bf16_tflops_sustained"]
        traffic, tsrc = None, None
        for name in ("conv_traffic_r2.json", "conv_traffic_r1.json"):
            tpath = os.path.join(ROOT, "profiles", name)
            if os.path.exists(tpath) and cfg["denoiser"] == "fastdvd_color" and c == 4:
                traffic, tsrc = json.load(open(tpath))["dram_bytes_per_launch"], "profiles/" + name    # ncu --set full capture, per launch
                break
        half_chain = cfg["denoiser"] == "fastdvd_color" or getattr(eng, "layers_h", None) is not None
        kind = "kind::f16" if half_chain else "kind::tf32"
        roofline = {"bound": "tensor", "kernel": "conv_fwd2_tc_kernel / conv_fwd_tc_kernel (tcgen05.mma %s)" % kind, "achieved": achieved,
                    "peak": peak_bf16, "unit": "TFLOP/s", "frac": achieved / peak_bf16, "traffic": traffic, "traffic_source": tsrc,
                    "peak_kind": pk_kind + " cuBLAS bf16 (sustained)" + ("; fp16 operands run at the bf16 rate" if kind == "kind::f16"
                                                                        else "; TF32 operands run at half the bf16 rate"),
                    "frac_of_operand_rate": achieved / (peak_bf16 if kind == "kind::f16" else peak_bf16 / 2),
                    "flops_per_pass": flops, "launches_per_pass": len(prof), "avg_launch_ms": 1e3 * conv_s / len(prof),
                    "timing": "CUDA events around %d back-to-back passes on the launching stream (as the solver runs them)" % n_pass,
                    "achieved_with_an_event_pair_per_launch": flops / conv_s_serial / 1e12,
                    "pass": "one inference pass over %dx%dx%d (algorithmic flops, temp1 evaluated once per frame)" % (bb, hh, W)}
        if cfg["denoiser"].startswith("ffdnet"):
            # FFDNet returns the image itself, so its convolutions run at ~fp32 accuracy: 3 tensor-core products per algorithmic one
            roofline["executed_products_per_flop"] = 3
            roofline["frac_executed"] = 3 * roofline["frac_of_operand_rate"]
        del u
    hbm_rows = hbm_kernel_table(min(H, 1024) if c == 5 else H, W, B, dev, pk["hbm_gbs"])
    roofline_hbm = {"peak": pk["hbm_gbs"], "unit": "GB/s", "peak_kind": pk_kind + " copy bandwidth",
                    "size": "%dx%dx%d" % (min(H, 1024) if c == 5 else H, W, B), "kernels": hbm_rows,
                    "note": "TV is instruction-bound (5 fused inner iterations on chip, IEEE sqrt/divide), see profiles/"}
    if roofline is None:                                                   # config 1: the TV kernel is the dominant one
        r = [x for x in hbm_rows if x["kernel"].startswith("tv")][0]
        roofline = {"bound": "hbm", "kernel": "tv_chambolle2_kernel (+ clip + dual update)", "achieved": r["achieved"],
                    "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": r["frac"], "traffic": None,
                    "peak_kind": pk_kind + " copy bandwidth", "avg_launch_ms": r["ms"]}
    # ---- delta PSNR against the REFERENCE's own output (tests/golden/fullsize.npz), configs 3 and 4, N = 1
    dpsnr = None
    gpath = os.path.join(ROOT, "tests", "golden", "fullsize.npz")
    if world == 1 and c in (3, 4) and not args.no_delta_psnr and os.path.exists(gpath):
        g = np.load(gpath)
        key = "c%d" % c
        reset_model()
        worker_init_fn(0)
        w_full = admm_denoise_bayer_demosaic_pre(meas, mask, 1, 0.01, 'tv', [40], False, [0], x0_bayer=None, X_orig=orig,
                                                 show_iqa=False)
        kw = dict(update_times=-1) if c == 4 else {}
        r = twoStageAdmm_denoise_bayer(meas, mask, 1, 0.01, cfg["denoiser"], cfg["iters"], False, cfg["sigma"],
                                       x0_bayer=torch.from_numpy(w_full[0]).cuda(), X_orig=orig, model_denoise=model,
                                       show_iqa=True, lr_=LR, interval_iter=cfg["interval"], logf=io.StringIO(), update_=True,
                                       update_per_iter=UPDATE_PER_ITER, **kw)
        s = int(g["shape"][4])
        dpsnr = {"value": float(np.mean(r[2]) - np.mean(g[key + "_psnr"])), "unit": "dB", "psnr_ours": float(np.mean(r[2])),
                 "psnr_reference": float(np.mean(g[key + "_psnr"])),
                 "max_abs_diff": float(np.max(np.abs(r[1][::s, ::s] - g[key + "_x_s"]))),
                 "max_abs_psnr_all_diff": float(np.max(np.abs(np.array(r[4]) - g[key + "_psnr_all"]))),
                 "against": "the reference's own CPU output for the same inputs (stage 1 + stage 2, tests/golden/fullsize.npz; "
                            "max_abs_diff over its strided sample)",
                 "note": "with the synthetic contractive FastDVDnet init the denoiser lowers the PSNR of the warm start in the "
                         "reference as well (trained weights are absent upstream)" if c == 4 else None}
    # ---- baselines
    cpu = None
    if not args.no_cpu_baseline and world == 1:          # the CPU leg is an N = 1 figure (rank 0's host cores); not repeated per N
        ref = CpuReference(c)
        t_inf = ref.inference_iter()
        t = ref.schedule_seconds(t_inf)
        cpu = {"value": n_iter / t, "unit": "iters/s", "sec_per_recon": t, "cores": ref.cores, "kind": "port", "sample": ref.describe()}
    eager = None
    if not args.no_gpu_eager and world == 1:
        if c == 5:
            eager = gpu_eager_baseline(c, cfg, meas_f, mask_f, orig_f, warm_f)
        else:
            eager = gpu_eager_baseline(c, cfg, meas, mask, orig, warm)
    line = {"metric": "admm_iters_per_sec", "value": value, "unit": "iters/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "sec_per_recon": ms * 1e-3 / args.steps,
            "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None,
            "dtype": {"tv": "f32", "fastdvd_color": "f16 operands / f32 accumulate (inference convs); tf32 / f32 (online update); f32 elsewhere",
                      "ffdnet_color": "tf32 (3-product split) / f32", "ffdnet_gray": "tf32 (3-product split) / f32"}[cfg["denoiser"]],
            "data": "synthetic",
            "config": config_dict(c, cfg), "clocks": clk,
            "e2e": {"value": e2e_value, "unit": "iters/s", "sec_per_recon": ms_e2e * 1e-3 / args.steps,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": launches, "roofline": roofline, "roofline_hbm": roofline_hbm, "cpu_baseline": cpu,
            "gpu_eager_baseline": eager, "delta_psnr": dpsnr}
    _emit(line)
    if world > 1:
        dist.destroy_process_group()


def _emit(line):
    """The ONE JSON line of the contract goes to the real stdout; everything else this process (or NCCL, which logs
    its version banner to stdout when NCCL_DEBUG is set) prints is routed to stderr."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)

if __name__ == "__main__":
    main()
