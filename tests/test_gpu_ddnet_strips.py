"""GPU: DDnet on row strips and in frame chunks reproduces the whole-frame engine bit for bit.

One process: the strips of a global frame are run one after another, their halo exchanges simulated by slicing the whole
frame's tensors (the mosaic, and for the temp2 input the un-tiled engine's own rows of the same frame chunk; every strip's
own rows of that input are checked against them on the way).  Two processes on the one GPU: stage 2 with ``model_demosaic``
(and with ``close_form_demosaic``) over strips equals the un-tiled solver."""
import io
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
H, W, B = 384, 40, 5          # 384 = 2 x 192 = 3 x 128 = 4 x 96 rows; W = 40 is not a multiple of the 128-pixel tile


def _ddnet():
    from adaptivepnp_sci_b200.network_demosaicking import DDnet
    from adaptivepnp_sci_b200.synthetic import ddnet_synthetic_state_dict
    m = DDnet()
    m.load_state_dict(ddnet_synthetic_state_dict(), strict=True)
    return m.eval().cuda()


def _mosaic():
    g = torch.Generator().manual_seed(11)
    return torch.rand(B, H, W, generator=g).cuda()


class _SlicedTile:
    """TileContext stand-in for strip ``rank`` of ``world``: exchange() cuts the extended strip out of the whole frame."""

    def __init__(self, rank, world, globals_):
        from adaptivepnp_sci_b200 import parallel
        self.rank, self.world, self.H_total, self.W = rank, world, H, W
        self.rows = H // world
        self.r0 = rank * self.rows
        self.globals = list(globals_)          # [mosaic [B,1,H,W], t2in of chunk 0 [2bc,1,H,32W], chunk 1, ...]
        self.own_equal = []
        self.halo_sizes = lambda halo: parallel.TileContext.halo_sizes(self, halo)

    def exchange(self, own, halo):
        full = self.globals.pop(0)
        assert full.shape[:2] == own.shape[:2] and full.shape[3] == own.shape[3]
        self.own_equal.append(bool(torch.equal(own, full[:, :, self.r0:self.r0 + self.rows])))
        top, bot = self.halo_sizes(halo)
        return full[:, :, self.r0 - top:self.r0 + self.rows + bot].contiguous(), top


def _untiled_t2in(eng, mosaic, Bc):
    """The un-tiled temp2 input of every frame chunk, [2bc,1,H,32W] each."""
    eng.prepare()
    out = []
    for f0 in range(0, B, Bc):
        bc = min(Bc, B - f0)
        t2in, _, _ = eng._stage_a(mosaic, f0, bc, Bc, 0, H, False)
        out.append(t2in.clone().view(2 * bc, 1, H, 32 * W))
    return out


def _tiled(eng, mosaic, world, Bc):
    res, own_ok = [], []
    t2 = _untiled_t2in(eng, mosaic, Bc)
    for r in range(world):
        t = _SlicedTile(r, world, [mosaic.view(B, 1, H, W)] + t2)
        own = mosaic[:, t.r0:t.r0 + t.rows].contiguous()
        res.append(eng.forward_tiled(own, t).clone())
        assert not t.globals                   # one mosaic exchange, one temp2-input exchange per chunk
        own_ok.append(all(t.own_equal))
    return torch.cat(res, dim=2), own_ok


@pytest.mark.parametrize("impl", ["ref", "tc"])
def test_strips_equal_whole_frame(cuda, monkeypatch, impl):
    monkeypatch.setenv("SCI_CONV_IMPL", impl)
    eng = _ddnet().engine()
    mosaic = _mosaic()
    ref = eng.forward(mosaic).clone()
    for world in (2, 3, 4):
        got, own_ok = _tiled(eng, mosaic, world, eng.tiled_chunk_frames(B, _SlicedTile(0, world, [])))
        assert all(own_ok), "strip %s: own rows of the temp2 input differ from the whole frame's" % own_ok
        assert torch.equal(got, ref), "%d strips: max |d| = %g" % (world, float((got - ref).abs().max()))


@pytest.mark.parametrize("which", ["STAGE_A_HALO", "STAGE_B_HALO"])
def test_smaller_halo_changes_own_rows(cuda, monkeypatch, which):
    monkeypatch.setenv("SCI_CONV_IMPL", "ref")
    eng = _ddnet().engine()
    mosaic = _mosaic()
    ref = eng.forward(mosaic).clone()
    monkeypatch.setattr(type(eng), which, 80 if which == "STAGE_A_HALO" else 32)
    got, _ = _tiled(eng, mosaic, 2, B)
    assert not torch.equal(got, ref)


@pytest.mark.parametrize("impl", ["ref", "tc"])
def test_frame_chunks_equal_one_pass(cuda, monkeypatch, impl):
    monkeypatch.setenv("SCI_CONV_IMPL", impl)
    eng = _ddnet().engine()
    mosaic = _mosaic()
    assert eng.chunk_frames(B, H, W) == B          # the default budget keeps such a frame in one pass
    ref = eng.forward(mosaic).clone()
    for Bc in (1, 2, 3, B):                        # 2 and 3 leave a ragged last chunk
        monkeypatch.setattr(type(eng), "PASS_PIXELS", 3 * Bc * H * W)
        assert eng.chunk_frames(B, H, W) == Bc
        assert torch.equal(eng.forward(mosaic), ref), "Bc = %d" % Bc
    monkeypatch.setattr(type(eng), "PASS_PIXELS", 2 * 3 * H * W)
    got, own_ok = _tiled(eng, mosaic, 3, 2)        # chunks of 2, 2, 1 on strips
    assert all(own_ok) and torch.equal(got, ref)


def test_upsample_strip_matches_whole_frame(cuda):
    """sci_ddnet_upsample4_strip on the rows a strip holds == sci_ddnet_upsample4 of the whole frame on its interior rows,
    with every buffer inside NaN sentinels, so a read outside the held rows would show up as a NaN."""
    from adaptivepnp_sci_b200._lib import call, ptr, stream
    g = torch.Generator().manual_seed(5)
    Bf, Hf, Wf, cp = 3, 64, 24, 32
    mosaic = torch.rand(Bf, Hf, Wf, generator=g).cuda()
    a2 = (0.5 + torch.rand(36, generator=g)).cuda()
    xo4 = torch.rand(3 * Bf, Hf // 2, Wf // 2, cp, generator=g).cuda()
    whole = torch.empty(3 * Bf, Hf, Wf, 32, device="cuda")
    call("sci_ddnet_upsample4", ptr(mosaic), ptr(a2), ptr(xo4), cp, ptr(whole), Bf, Hf, Wf, 32, 0, stream())

    def fenced(t, pad=4096):
        buf = torch.full((t.numel() + 2 * pad,), float("nan"), device="cuda")
        buf[pad:pad + t.numel()] = t.reshape(-1)
        return buf, buf[pad:pad + t.numel()].view(t.shape)

    for f0, Bc in ((0, Bf), (1, 2), (2, 1)):
        for row0, rows in ((0, 16), (16, 24), (40, 24), (8, 56)):
            _, m_s = fenced(mosaic[:, row0:row0 + rows].contiguous())
            # xo4 of the chunk only (batch j*Bc + f-f0, as the engine's temp11 pass of that chunk produces it)
            x_chunk = xo4.view(3, Bf, Hf // 2, Wf // 2, cp)[:, f0:f0 + Bc].reshape(3 * Bc, Hf // 2, Wf // 2, cp)
            _, x_s = fenced(x_chunk[:, row0 // 2:(row0 + rows) // 2].contiguous())
            ob, o_s = fenced(torch.zeros(3 * Bc, rows, Wf, 32, device="cuda"))
            call("sci_ddnet_upsample4_strip", ptr(m_s), ptr(a2), ptr(x_s), cp, ptr(o_s), Bf, f0, Bc, rows, Wf, row0, Hf, 32, 0,
                 stream())
            torch.cuda.synchronize()
            assert torch.isnan(ob).sum() == 2 * 4096                 # the fences are intact and nothing read outside
            want = whole.view(3, Bf, Hf, Wf, 32)[:, f0:f0 + Bc, row0:row0 + rows].reshape(3 * Bc, rows, Wf, 32)
            lo = 0 if row0 == 0 else 2                               # rows whose sources the strip holds
            hi = rows if row0 + rows == Hf else rows - 2
            assert torch.equal(o_s[:, lo:hi], want[:, lo:hi]), (f0, Bc, row0, rows)


# ---- two processes: the solver over strips ---------------------------------------------------------------------------
SH, SW, SB = 352, 32, 3        # 2 strips of 176 rows
KW = dict(show_iqa=True, demosaic_method='malvar2004', lr_=2e-6, interval_iter=2, update_=True, update_per_iter=1)


def _case():
    from adaptivepnp_sci_b200.synthetic import make_case
    meas, mask, orig = make_case(SH, SW, SB, 77, bayer=True)
    warm = np.clip(meas[:, :, None] * mask / np.maximum(mask.sum(2, keepdims=True), 1), 0, 1).astype(np.float32)
    return meas, mask, orig, warm


def _denoiser(name):
    if name == 'ffdnet_color':
        from adaptivepnp_sci_b200.network_ffdnet import FFDNet
        m = FFDNet(3, 3, 96, 12, 'R')
        m.load_state_dict(torch.load(os.path.join(ROOT, "model_zoo", "ffdnet_color.pth")), strict=True)
        return m.eval().cuda()
    from adaptivepnp_sci_b200.fastdvdnet_adapter import DataParallelLike
    from adaptivepnp_sci_b200.fastdvdnet_models import FastDVDnet
    from adaptivepnp_sci_b200.synthetic import fastdvdnet_synthetic_state_dict
    m = DataParallelLike(FastDVDnet())
    m.load_state_dict({"module." + k: v for k, v in fastdvdnet_synthetic_state_dict().items()}, strict=True)
    return m.eval().cuda()


def _solve(name, deep, close_form, tile=None):
    from adaptivepnp_sci_b200.dvp_linear_inv_2_stage_ADMM_tensor_online import twoStageAdmm_denoise_bayer
    from adaptivepnp_sci_b200.utilspy import worker_init_fn
    meas, mask, orig, warm = _case()
    sl = tile.slice_rows if tile is not None else (lambda a: a)
    m = _denoiser(name)
    worker_init_fn(0)
    r = twoStageAdmm_denoise_bayer(sl(meas), sl(mask), 1, 0.01, name, [4], False, [12 / 255],
                                   x0_bayer=torch.from_numpy(sl(warm)).cuda(), X_orig=sl(orig), model_denoise=m,
                                   model_demosaic=_ddnet() if deep else None, close_form_demosaic=close_form,
                                   logf=io.StringIO(), tile=tile, update_times=-1, **KW)
    return r[0], r[1], np.array(r[4])


def _worker(rank, world, port, q, name, deep, close_form):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK="0", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port),
                      SCI_CONV_IMPL="ref")
    from adaptivepnp_sci_b200 import parallel
    ctx = parallel.init(backend="gloo")
    tile = parallel.TileContext(ctx, SH, SW)
    rgb, xb, psnr_all = _solve(name, deep, close_form, tile)
    q.put((rank, rgb, xb, psnr_all, tile.p2p is not None))
    ctx.finalize()


@pytest.mark.parametrize("name,deep,close_form", [("ffdnet_color", True, False), ("fastdvd_color", True, False),
                                                  ("ffdnet_color", False, True), ("fastdvd_color", True, True)])
def test_tiled_stage2_deep_demosaic_equals_untiled(cuda, monkeypatch, name, deep, close_form):
    """DDnet (88-row mosaic halo, 40-row temp2-input halo) and the pixel-wise closed form over 2 strips, inference
    iterations and one online update of the denoiser: the un-tiled result within the tolerances of test_gpu_tiled.py."""
    monkeypatch.setenv("SCI_CONV_IMPL", "ref")
    ref = _solve(name, deep, close_form)
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctxm = mp.get_context("spawn")
    q = ctxm.Queue()
    procs = [ctxm.Process(target=_worker, args=(r, 2, port, q, name, deep, close_form)) for r in range(2)]
    for p in procs:
        p.start()
    outs = sorted((q.get(timeout=300) for _ in range(2)), key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, rgb, xb, psnr_all, used_p2p in outs:
        assert used_p2p
        assert rgb.shape == (SH, SW, 3, SB) and xb.shape == (SH, SW, SB)
        assert np.max(np.abs(rgb - ref[0])) < 2e-5 and np.max(np.abs(xb - ref[1])) < 2e-5
        assert np.max(np.abs(psnr_all - ref[2])) < 1e-3
