"""Micro-benchmark of single conv layers on the tensor-core kernels (CUDA events; inputs >> L2 or flushed).

    python tools/bench_conv.py            # FastDVDnet layer shapes at 512x512x8
    SCI_CONV_DBG=1|2|4 ...                # timing experiments of the v2 kernel: no MMAs / no activation loads / no stores
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from adaptivepnp_sci_b200 import engine

SHAPES = [   # N, H, W, Ci, Co, stride, ps
    (8, 512, 512, 12, 90, 1, False), (8, 512, 512, 90, 32, 1, False), (8, 512, 512, 32, 32, 1, False),
    (8, 512, 512, 32, 3, 1, False), (8, 256, 256, 64, 64, 1, False), (8, 128, 128, 128, 128, 1, False),
    (8, 256, 256, 64, 128, 1, True), (8, 128, 128, 128, 256, 1, True), (8, 512, 512, 32, 64, 2, False),
    (8, 256, 256, 64, 128, 2, False),
]


def main():
    dev = torch.device("cuda:0")
    eng = engine._EngineBase(torch.nn.Identity(), [])
    flush = torch.zeros(64 * 1024 * 1024, device=dev)
    for N, H, W, Ci, Co, stride, ps in SHAPES:
        conv = torch.nn.Conv2d(Ci, Co, 3, stride=stride, padding=1, bias=False).to(dev)
        L = engine.ConvLayer(conv, None, relu=True, stride=stride, ps=ps)
        engine.OpTable(L.fwd_ops(True), dev).run()
        x = torch.rand(N, H, W, L.Ci_pad, device=dev)
        Ho, Wo = (H // stride, W // stride) if not ps else (2 * H, 2 * W)
        y = torch.empty(N, Ho, Wo, L.out_ch, device=dev)
        for _ in range(3):
            eng.conv(L, x, N, H, W, y)
        ts = []
        for _ in range(10):
            flush.add_(1.0)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            eng.conv(L, x, N, H, W, y)
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        ts.sort()
        ms = ts[len(ts) // 2]
        fl = 2.0 * N * (H // stride) * (W // stride) * 9 * Ci * Co
        by = 4.0 * (x.numel() + y.numel())
        # weight gradient of the same layer (dz has the GEMM-output shape [N, H/stride, W/stride, Co_pad])
        eng.layers = [L]
        L.dwpk = torch.zeros(9 * L.Co_pad * L.Ci_pad, device=dev)
        L.scale = None
        dz = torch.rand(N, H // stride, W // stride, L.Co_pad, device=dev)
        for _ in range(3):
            eng.wgrad(L, x, dz, N, H, W)
        tw = []
        for _ in range(10):
            flush.add_(1.0)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            eng.wgrad(L, x, dz, N, H, W)
            b.record()
            torch.cuda.synchronize()
            tw.append(a.elapsed_time(b))
        tw.sort()
        mw = tw[len(tw) // 2]
        print("%4dx%-4d %3d->%-3d s%d ps%d  fwd %.4f ms %7.1f TFLOP/s(alg) %6.0f GB/s | wgrad %.4f ms %7.1f TFLOP/s(alg)" %
              (H, W, Ci, Co, stride, int(ps), ms, fl / ms / 1e9, by / ms / 1e6, mw, fl / mw / 1e9))


main()
