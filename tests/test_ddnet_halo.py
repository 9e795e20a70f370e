"""CPU: the row halos of DDnet on strips (engine.DDnetEngine.STAGE_A_HALO / STAGE_B_HALO) cover its receptive field, and
strips DDnet cannot run on are refused before any GPU work.

Receptive field: the float64 oracle DDnet with positive weights and inputs (nothing cancels, every ReLU passes), on a
1024-row frame; for output rows near the top, the middle and the bottom, the rows of the input whose gradient is nonzero.
The bilinear up-sampling of path 2 (align_corners=True) lags its source row by up to one full-resolution row towards the
bottom of the frame, so the probe covers both ends."""
import types

import pytest
import torch

H, W = 1024, 16
ROWS = (8, 100, 515, 930, 1019)


def _positive(module, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for p in module.parameters():
            p.copy_(0.02 + 0.1 * torch.rand(p.shape, generator=g, dtype=torch.float64))
    return module


def _support(out_fn, leaves, r):
    """Rows of the leaves that output row r depends on, relative to r."""
    for t in leaves:
        t.grad = None
    out_fn()[..., r, :].sum().backward()
    rows = torch.zeros(H, dtype=torch.bool)
    for t in leaves:
        rows |= (t.grad.abs().sum(dim=tuple(i for i in range(t.dim()) if i != t.dim() - 2)) > 0)
    idx = torch.nonzero(rows).flatten()
    return int(idx.min()) - r, int(idx.max()) - r


@pytest.fixture(scope="module")
def supports():
    from oracle.networks import DDnet, _mosaic_to_4ch
    torch.manual_seed(0)
    net = _positive(DDnet().double(), 1)
    fr = [torch.rand(1, H, W, dtype=torch.float64, requires_grad=True) for _ in range(5)]
    a, a2 = net.weight_tensor_in, net.weight_tensor_in2

    def path1():
        return net.temp1(*(fr[k].unsqueeze(1) * a[k] for k in range(3)))

    def path2():
        return net.temp11(*(_mosaic_to_4ch(fr[k]) * a2[k] for k in range(3)))

    t2in = [torch.rand(1, 3, H, W, dtype=torch.float64, requires_grad=True) for _ in range(3)]
    res = {}
    for r in ROWS:
        res[r] = dict(path1=_support(path1, fr[:3], r), path2=_support(path2, fr[:3], r),
                      temp2=_support(lambda: net.temp2(*t2in), t2in, r))
    return res


def _inside(lo_hi, r, halo):
    lo, hi = lo_hi
    return max(-halo, -r) <= lo and hi <= min(halo, H - 1 - r)


def test_stage_a_halo_covers_both_paths(supports):
    from adaptivepnp_sci_b200.engine import DDnetEngine
    for r, s in supports.items():
        assert _inside(s["path1"], r, DDnetEngine.STAGE_A_HALO), (r, s)
        assert _inside(s["path2"], r, DDnetEngine.STAGE_A_HALO), (r, s)


def test_stage_b_halo_covers_temp2(supports):
    from adaptivepnp_sci_b200.engine import DDnetEngine
    for r, s in supports.items():
        assert _inside(s["temp2"], r, DDnetEngine.STAGE_B_HALO), (r, s)


def test_path2_needs_more_than_80_rows(supports):
    """Teeth: away from the frame's edges path 2 reaches past 80 rows, so the next smaller multiple of 8 would not do."""
    mid = [s["path2"] for r, s in supports.items() if 100 <= r <= 930]
    assert max(max(-lo, hi) for lo, hi in mid) > 80
    assert max(max(-lo, hi) for lo, hi in (s["temp2"] for s in supports.values())) > 32


class _Tile(types.SimpleNamespace):
    pass


@pytest.mark.parametrize("rows,W_,world", [(84, 64, 2), (100, 64, 2), (96, 60, 2), (80, 64, 4)])
def test_refused_strips(rows, W_, world):
    """Strips not a multiple of 8 rows, a width not a multiple of 8, strips shorter than the 88-row halo: ValueError
    from the solver before it touches the inputs."""
    from adaptivepnp_sci_b200.dvp_linear_inv_2_stage_ADMM_tensor_online import twoStageAdmm_denoise_bayer
    from adaptivepnp_sci_b200.engine import DDnetEngine
    tile = _Tile(rows=rows, W=W_, world=world, rank=0, H_total=rows * world, r0=0)
    with pytest.raises(ValueError):
        DDnetEngine.check_tile(tile)
    with pytest.raises(ValueError, match="DDnet on row strips"):
        twoStageAdmm_denoise_bayer(None, None, 1, 0.01, 'ffdnet_color', [1], False, [0.1], model_demosaic=object(),
                                   tile=tile)


def test_accepted_strips():
    from adaptivepnp_sci_b200.engine import DDnetEngine
    DDnetEngine.check_tile(_Tile(rows=88, W=40, world=8, rank=0, H_total=704, r0=0))
    DDnetEngine.check_tile(_Tile(rows=48, W=40, world=1, rank=0, H_total=48, r0=0))      # one rank: no halo needed


def test_chunk_frames():
    from adaptivepnp_sci_b200.engine import DDnetEngine
    P = DDnetEngine.PASS_PIXELS
    assert DDnetEngine.chunk_frames(8, 512, 512) == 8                   # sizes of the single-GPU runs: one pass
    for B, Hh, Ww in ((24, 432, 2048), (24, 2048, 2048), (7, 1024, 1024), (24, 336, 2048)):
        bc = DDnetEngine.chunk_frames(B, Hh, Ww)
        n = -(-B // bc)
        assert 3 * bc * Hh * Ww <= P or bc == 1
        assert n == -(-B // max(1, P // (3 * Hh * Ww)))                 # no more chunks than the budget asks for
    tile = _Tile(rows=256, W=2048, world=8, rank=7, H_total=2048, r0=1792)
    assert DDnetEngine.tiled_chunk_frames(24, tile) == DDnetEngine.chunk_frames(24, 256 + 176, 2048)
