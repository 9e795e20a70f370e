"""The TV prior on row strips of one frame (sci_tv_strip_main / _finish, sci_halo_send_tv, TileContext.tv_chambolle).

Every own pixel of a strip is computed from the same inputs in the same order as by the un-tiled kernel, so theta and
b_out must be bit-identical whenever the stop decisions agree; the decisions agree on these inputs (they could differ only
where |E_prev - E_k| - eps*E_init is within fp64 rounding of zero, the energies being summed in another order).

The argument checks at the end need no GPU."""
import ctypes
import io
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _stack4_to_planar(stack4, dev):
    from oracle import sci_ops
    from adaptivepnp_sci_b200 import ops
    hwb = sci_ops.fourCh2OneCh(torch.from_numpy(np.ascontiguousarray(stack4))).contiguous().to(dev)
    H, W, B = hwb.shape
    return ops.pixlast_to_planar(hwb, 1, B).view(B, H, W)


def _frame(H, W, B, band, seed):
    """[h, w, B+2, 4] channel stack: mixed noise amplitudes (stops at 1, 3 and 4), one nearly flat frame, and one frame whose
    rows [band) carry sigma-50 noise and the others sigma 8 (its stop depends on which strips' energies are summed)."""
    rng = np.random.default_rng(seed)
    h, w = H // 2, W // 2
    yy, xx = np.mgrid[0:h, 0:w]
    stack = np.empty((h, w, B + 2, 4), np.float32)
    for t in range(B):
        for ib in range(4):
            noise = (0.08, 8.0, 50.0)[(t + ib) % 3] * rng.standard_normal((h, w))
            stack[:, :, t, ib] = 0.5 + 0.3 * np.sin((xx + 3 * t) / 9.0) * np.cos((yy + ib) / 7.0) + noise
    stack[:, :, B] = 0.5 + 0.02 * rng.random((h, w, 4))
    inband = (yy >= band[0] // 2) & (yy < band[1] // 2)
    for ib in range(4):
        stack[:, :, B + 1, ib] = (0.5 + 0.3 * np.sin(xx / 9.0) * np.cos((yy + ib) / 7.0)
                                  + np.where(inband, 50.0, 8.0) * rng.standard_normal((h, w)))
    return stack


def _run_strips(x, b, c_b, s_b, clip, strips, cut=None, drop=None):
    """Cut x [B, H, W] (and b) into strips, halos filled from the full frame's f = x + c_b*b (numpy float32), main pass per
    strip, esums stacked in strip order (``drop``: leave one strip's out), finish per strip.  Returns the assembled theta,
    b_out and the per-strip nstop.  ``cut``: (strip index, rows) keeps only the nearest rows of that strip's top halo."""
    from adaptivepnp_sci_b200 import ops
    B, H, W = x.shape
    xn = x.cpu().numpy()
    f = xn if b is None else xn + np.float32(c_b) * b.cpu().numpy()
    theta, b_out = torch.full_like(x, np.nan), (torch.full_like(x, np.nan) if b is not None else None)
    runs, r0 = [], 0
    for i, rows in enumerate(strips):
        xs = x[:, r0:r0 + rows].contiguous()
        bs = b[:, r0:r0 + rows].contiguous() if b is not None else None
        ht = torch.from_numpy(np.ascontiguousarray(f[:, r0 - 8:r0])).to(x.device) if r0 > 0 else None
        hb = torch.from_numpy(np.ascontiguousarray(f[:, r0 + rows:r0 + rows + 8])).to(x.device) if r0 + rows < H else None
        if cut is not None and cut[0] == i:
            ht[:, :8 - cut[1]] = 0
        th, bo = torch.empty_like(xs), (torch.empty_like(xs) if b is not None else None)
        ws = ops.TvStripWorkspace(rows, W, B, x.device)
        esum = ops.tv_strip_main(xs, bs, c_b, th, bo, s_b, clip, ws, r0, H, ht, hb).clone()
        runs.append((r0, rows, xs, bs, ht, hb, th, bo, ws, esum))
        r0 += rows
    esum_all = torch.stack([r[-1] for i, r in enumerate(runs) if i != drop]).contiguous()
    nstops = []
    for r0, rows, xs, bs, ht, hb, th, bo, ws, _ in runs:
        ns = torch.full((4 * B,), -1, dtype=torch.int32, device=x.device)
        ops.tv_strip_finish(xs, bs, c_b, th, bo, s_b, clip, ws, r0, H, esum_all, ht, hb, nstop_out=ns)
        theta[:, r0:r0 + rows] = th
        if b is not None:
            b_out[:, r0:r0 + rows] = bo
        nstops.append(ns.cpu().numpy())
    return theta, b_out, nstops


# ragged in both directions: W = 130 / 76 (three / two 64-column tiles, the last partial), strips of 8 .. 100 rows, none a
# multiple of the 32-row tile; the sigma-50 band is the 100-row strip
@gpu
@pytest.mark.parametrize("W,strips", [(130, (8, 12, 36, 100)), (76, (100, 36, 12, 8))])
def test_strips_equal_untiled(cuda, W, strips):
    from adaptivepnp_sci_b200 import ops
    from oracle import tv_chambolle
    H, B = sum(strips), 2
    big = strips.index(100)
    band = (sum(strips[:big]), sum(strips[:big]) + 100)
    stack = _frame(H, W, B, band, seed=W)
    Bt = B + 2
    _, stops = tv_chambolle.denoise_tv_chambolle(stack.reshape(H // 2, W // 2, 4 * Bt), 0.1, n_iter_max=5,
                                                 multichannel=True, return_stops=True)
    want_stops = np.minimum(np.array(stops), 4)
    x = _stack4_to_planar(stack, cuda)
    g = torch.Generator(device=cuda).manual_seed(W)
    bb = 0.05 * torch.randn(x.shape, generator=g, device=cuda)
    ws = ops.TvWorkspace(H, W, Bt, cuda)
    for b, c_b, s_b, clip in [(None, 0.0, 0.0, False), (bb, -1.0, -1.0, True)]:
        theta_ref = torch.empty_like(x)
        b_ref = torch.empty_like(x) if b is not None else None
        nstop_ref = torch.zeros(4 * Bt, dtype=torch.int32, device=cuda)
        ops.tv_chambolle(x, b, c_b, theta_ref, b_ref, s_b, clip, ws, nstop_out=nstop_ref)
        nstop_ref = nstop_ref.cpu().numpy()
        theta, b_out, nstops = _run_strips(x, b, c_b, s_b, clip, strips)
        for ns in nstops:
            assert np.array_equal(ns, nstop_ref), (ns, nstop_ref)
        assert torch.equal(theta, theta_ref)
        if b is None:
            assert np.array_equal(nstop_ref, want_stops), (nstop_ref, want_stops)
            assert (want_stops == 1).any() and (want_stops == 3).any() and (want_stops == 4).any()
        else:
            assert torch.equal(b_out, b_ref)
            assert (nstop_ref < 4).any()                  # the fix-up pass rewrote channels that stopped early
        # teeth: a top halo cut to its 6 nearest rows changes the rows next to that boundary ...
        k = 2 if strips[0] == 8 else 1
        r0 = sum(strips[:k])
        theta_cut, _, _ = _run_strips(x, b, c_b, s_b, clip, strips, cut=(k, 6))
        assert not torch.equal(theta_cut[:, r0:r0 + 8], theta_ref[:, r0:r0 + 8])
        # ... and the decision without the 100-row strip's energies is a different one
        _, _, nstops_drop = _run_strips(x, b, c_b, s_b, clip, strips, drop=big)
        assert not np.array_equal(nstops_drop[0], nstop_ref)


@gpu
def test_halo_send_tv_stores_f(cuda):
    """sci_halo_send_tv with this device's own buffers standing in for the neighbours' slots: the boundary rows of
    f = x + c_b*b, rounded as numpy float32 rounds them, and the sequence number in both flag words."""
    from adaptivepnp_sci_b200 import ops
    B, rows, W = 3, 20, 18
    g = torch.Generator(device=cuda).manual_seed(1)
    x = torch.rand((B, rows, W), generator=g, device=cuda)
    b = torch.randn((B, rows, W), generator=g, device=cuda)
    up, down = torch.full((B, 8, W), np.nan, device=cuda), torch.full((B, 8, W), np.nan, device=cuda)
    flags = torch.zeros(3, dtype=torch.int32, device=cuda)          # up flag, down flag, done counter
    ops.halo_send_tv(x, b, 0.7, up.data_ptr(), down.data_ptr(), flags.data_ptr(), flags.data_ptr() + 4, 5,
                     flags.data_ptr() + 8)
    f = x.cpu().numpy() + np.float32(0.7) * b.cpu().numpy()
    assert np.array_equal(up.cpu().numpy(), f[:, :8]) and np.array_equal(down.cpu().numpy(), f[:, rows - 8:])
    assert flags.cpu().tolist() == [5, 5, 0]
    ops.halo_send_tv(x, None, 0.0, None, down.data_ptr(), None, flags.data_ptr() + 4, 6, flags.data_ptr() + 8)
    assert np.array_equal(down.cpu().numpy(), x.cpu().numpy()[:, rows - 8:]) and flags.cpu().tolist() == [5, 6, 0]


def _case(H, W, B, seed):
    from adaptivepnp_sci_b200.synthetic import make_case
    return make_case(H, W, B, seed, bayer=True)


@gpu
def test_single_strip_equals_untiled(cuda):
    """world = 1: TileContext.tv_chambolle gives the bits of ops.tv_chambolle, nstop included, over a whole stage-1 run."""
    from adaptivepnp_sci_b200 import ops, parallel
    from adaptivepnp_sci_b200.dvp_linear_inv_2_stage_ADMM_tensor_online import _Problem
    H, W, B = 96, 80, 3
    meas, mask, _ = _case(H, W, B, 21)
    tile = parallel.TileContext(parallel.Context(0, 1, 0, "gloo"), H, W)
    pbs = [_Problem(meas, mask, None, None) for _ in range(2)]
    wss = [ops.TvWorkspace(H, W, B, cuda), ops.TvStripWorkspace(H, W, B, cuda)]
    tvs = [ops.tv_chambolle, tile.tv_chambolle]
    bns = [torch.empty_like(pbs[0].b) for _ in range(2)]
    seen = set()
    for k in range(40):
        out = []
        for i in range(2):
            pb = pbs[i]
            ops.project_stage1(pb.theta, pb.b, pb.phi, pb.y, pb.phisum, pb.x, 1, 0.01)
            ns = torch.zeros(4 * B, dtype=torch.int32, device=cuda)
            tvs[i](pb.x, pb.b, -1.0, pb.theta, bns[i], -1.0, True, wss[i], nstop_out=ns)
            pb.b, bns[i] = bns[i], pb.b
            out.append((pb.x.clone(), pb.theta.clone(), pb.b.clone(), ns.cpu().numpy()))
        (x0, t0, b0, n0), (x1, t1, b1, n1) = out
        assert torch.equal(x0, x1) and torch.equal(t0, t1) and torch.equal(b0, b1) and np.array_equal(n0, n1), k
        seen.update(n0.tolist())
    assert len(seen) > 1                                  # early stops happened along the way


SH, SW, SB = 128, 64, 4


def _stage_runs(tile, sl):
    """Stage 1 ([40] TV iterations) -> stage 2 'tv' ([6]) from its warm start, from the host result and from the device
    strip.  ``sl`` cuts this rank's rows (identity when un-tiled)."""
    from adaptivepnp_sci_b200.dvp_linear_inv_2_stage_ADMM_tensor_online import (admm_denoise_bayer_demosaic_pre,
                                                                                twoStageAdmm_denoise_bayer)
    meas, mask, orig = _case(SH, SW, SB, 4242)
    kw = dict(X_orig=sl(orig), logf=io.StringIO(), tile=tile)
    s1 = admm_denoise_bayer_demosaic_pre(sl(meas), sl(mask), 1, 0.01, 'tv', [40], True, [None], **kw)
    x_dev = admm_denoise_bayer_demosaic_pre(sl(meas), sl(mask), 1, 0.01, 'tv', [40], True, [None], return_device=True,
                                            tile=tile)
    s2 = twoStageAdmm_denoise_bayer(sl(meas), sl(mask), 1, 0.01, 'tv', [6], False, [None], x0_bayer=sl(s1[0]), **kw)
    s2d = twoStageAdmm_denoise_bayer(sl(meas), sl(mask), 1, 0.01, 'tv', [6], False, [None], x0_bayer=x_dev, **kw)
    return s1, s2, s2d, x_dev.cpu().numpy()


def _worker(rank, world, port, q, p2p):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK="0", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port),
                      SCI_TILE_P2P=p2p)
    from adaptivepnp_sci_b200 import parallel
    ctx = parallel.init(backend="gloo")
    tile = parallel.TileContext(ctx, SH, SW)
    s1, s2, s2d, x_dev = _stage_runs(tile, tile.slice_rows)
    q.put((rank, s1, s2, s2d, x_dev, tile.p2p is not None))
    if tile.p2p is not None:
        tile.p2p.close()
    ctx.finalize()


@gpu
@pytest.mark.parametrize("p2p", ["1", "0"])
def test_two_strips_stage1_stage2_tv(cuda, p2p):
    """Two processes on one GPU (gloo; the halo goes through CUDA IPC peer to peer, or with SCI_TILE_P2P=0 through
    torch.distributed): stage 1 and stage-2 'tv' on two strips equal the un-tiled runs."""
    ref1, ref2, _, ref_x = _stage_runs(None, lambda a: a)
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctxm = mp.get_context("spawn")
    q = ctxm.Queue()
    procs = [ctxm.Process(target=_worker, args=(r, 2, port, q, p2p)) for r in range(2)]
    for p in procs:
        p.start()
    outs = sorted((q.get(timeout=300) for _ in range(2)), key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert np.array_equal(np.concatenate([o[4] for o in outs]), ref_x)     # return_device strips = the un-tiled x
    for rank, s1, s2, s2d, _, used_p2p in outs:
        assert used_p2p == (p2p == "1")
        assert len(s1) == 4 and len(s2) == 4
        assert np.array_equal(s1[0], ref1[0])                                 # x, bit for bit
        assert np.max(np.abs(np.array(s1[3]) - np.array(ref1[3]))) < 1e-6     # psnr_all
        assert np.max(np.abs(np.array(s1[1]) - np.array(ref1[1]))) < 1e-6     # per-frame PSNR
        assert np.max(np.abs(np.array(s1[2]) - np.array(ref1[2]))) < 1e-6     # per-frame SSIM
        assert np.array_equal(s2[0], ref2[0])                                 # stage-2 theta, bit for bit
        assert np.max(np.abs(np.array(s2[3]) - np.array(ref2[3]))) < 1e-6
        assert np.array_equal(s2d[0], s2[0])                                  # device warm start = host round trip
        # the PSNR sums add per-block fp64 partials atomically, so their last bits vary from run to run on equal images
        assert np.max(np.abs(np.array(s2d[3]) - np.array(s2[3]))) < 1e-9


# ---- refusals -------------------------------------------------------------------------------------------------------

def test_strip_shorter_than_halo_refused():
    from adaptivepnp_sci_b200 import ops, parallel
    tile = parallel.TileContext(parallel.Context(0, 2, 0, "gloo"), 8, 16)     # 4-row strips
    x = torch.zeros((1, 4, 16))
    with pytest.raises(ValueError, match="shorter than the 8-row halo"):
        tile.tv_chambolle(x, None, 0.0, x, None, 0.0, False, ws=None)
    assert ops.TV_HALO == 8


def test_tiled_stage1_deep_branch_refused():
    from adaptivepnp_sci_b200 import parallel
    from adaptivepnp_sci_b200.dvp_linear_inv_2_stage_ADMM_tensor_online import admm_denoise_bayer_demosaic_pre
    tile = parallel.TileContext(parallel.Context(0, 2, 0, "gloo"), 64, 16)
    for name in ('ffdnet_color', 'fastdvd_color'):
        with pytest.raises(NotImplementedError, match="deep stage-1 branches"):
            admm_denoise_bayer_demosaic_pre(np.zeros((32, 16), np.float32), np.zeros((32, 16, 2), np.float32), 1, 0.01,
                                            name, [2], tile=tile)


def test_strip_abi_refusals():
    """Every argument check runs before any CUDA call (so this runs without a GPU)."""
    from adaptivepnp_sci_b200 import _lib
    lib = _lib.lib
    P = ctypes.c_void_p(256)                          # never dereferenced: the checks fail first
    rows, W, B, H = 16, 64, 2, 48
    ws = ctypes.c_size_t(lib.sci_tv_strip_workspace_bytes(rows, W, B))
    assert ws.value > 0

    def main(row0=16, top=P, bot=P, n_iter_max=5, flag_top=None, err=None):
        return lib.sci_tv_strip_main(P, None, 0.0, P, None, 0.0, 0, rows, W, B, row0, H, top, bot, flag_top, None, 0, err,
                                     0.1, 2e-4, n_iter_max, P, ws, P, None)

    def finish(row0=16, top=P, bot=P, n_iter_max=5):
        return lib.sci_tv_strip_finish(P, None, 0.0, P, None, 0.0, 0, rows, W, B, row0, H, top, bot, 0.1, 2e-4, n_iter_max,
                                       P, ws, P, 2, None, None)

    for fn in (main, finish):
        assert fn(row0=15) == -1 and b"invalid argument" in lib.sci_last_error()          # odd row0
        assert fn(top=None) == -1 and b"halo" in lib.sci_last_error()                     # neighbour above, no halo
        assert fn(row0=32, bot=P) == -1                                                    # no neighbour below, yet a halo
        assert fn(n_iter_max=1) == -3 and b"n_iter_max" in lib.sci_last_error()            # SCI_EUNSUPPORTED
        assert fn(n_iter_max=6) == -3
    assert main(flag_top=P) == -1                                                           # a flag needs the error word
    assert lib.sci_tv_strip_main(P, None, 0.0, P, None, 0.0, 0, 6, W, B, 0, H, None, P, None, None, 0, None, 0.1, 2e-4, 5,
                                 P, ws, P, None) == -1                                       # rows < 8
    assert lib.sci_tv_strip_main(P, None, 0.0, P, None, 0.0, 0, rows, W, B, 16, H, P, P, None, None, 0, None, 0.1, 2e-4, 5,
                                 P, ctypes.c_size_t(ws.value - 8), P, None) == -4            # workspace too small
    # halo send: odd width, a slot without its flag word
    assert lib.sci_halo_send_tv(P, None, 0.0, B, rows, 63, 8, P, None, P, None, 1, P, None) == -1
    assert lib.sci_halo_send_tv(P, None, 0.0, B, rows, W, 8, P, None, None, None, 1, P, None) == -1
