"""GPU: the backward-pass reductions of the online update run in a fixed order, so a fine-tune is bit-reproducible.

Three reductions used to add with atomics in whatever order the CTAs finished: the weight gradient (every CTA's TMEM / FFMA
accumulator into the packed dW), the column sums fused into the data-gradient epilogue (bias / BatchNorm gradients) and
act_bwd's column sums.  Their ordered forms store one partial per CTA into a slot of a workspace and add the slots in slot
order in a second kernel of the same call.  Checked here:

* kernel contract, per weight-gradient plan (the plans tests/test_gpu_conv_plans.py forces, and the fp32 reference kernel),
  per fused column-sum case (with and without col_s2, PixelShuffle with one and two launches) and for act_bwd at ragged
  sizes: every slot is written, the result is fl(prefill + S) bit for bit with S the float32 left-to-right sum of the slots
  read back, summing the slots in reverse order gives other bits (so the check tells orders apart), two calls give the same
  bits, the result is within the float64 bound of the atomic form, and the non-reduced outputs (dz) equal the atomic form's;
* engines: one fine-tune call twice from the same weights and noise - weights, Adam moments and the output bit-identical
  (FastDVDnet colour / gray, FFDNet colour / gray, tensor-core and fp32 engines, a ragged batch of 7 frames);
* public entry points: the two solvers with online adaptation twice after worker_init_fn(0) - images and state_dict
  bit-identical;
* two processes on one GPU over gloo: a tiled FastDVDnet stage 2 with an online update, and a shared-weight fine-tune, each
  run twice - strips and weights bit-identical."""
import ctypes
import io
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp
import torch.nn.functional as F

from test_gpu_conv import _fastdvd, _ffdnet, impl  # noqa: F401  (impl: fixture, fp32 reference and tensor-core engines)
from test_gpu_conv_plans import C_ACC, KNOBS, WGRAD_CASES, tf32
from test_gpu_gray_fastdvd import _gray_model

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")


def _L():
    from adaptivepnp_sci_b200 import _lib
    return _lib


def _bits(t):
    return t.contiguous().view(torch.int32)


@pytest.fixture
def knobs(monkeypatch):
    """Kernel cases start from the planner's defaults and print their plans."""
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("SCI_CONV_VERBOSE", "1")
    return monkeypatch


def _check_slots(tag, part, prefill, got):
    """part [slots, n] read back from the workspace; got = the reduced output, prefill its value before the call."""
    assert part.shape[0] >= 2, "%s: %d slot(s) - nothing to order" % (tag, part.shape[0])
    assert bool(torch.isfinite(part).all()), "%s: slot elements left unwritten" % tag
    s = part[0].clone()
    for b in range(1, part.shape[0]):
        s = s + part[b]
    assert torch.equal(_bits(got), _bits(prefill + s)), "%s: not fl(prefill + left-to-right slot sum)" % tag
    r = part[-1].clone()
    for b in range(part.shape[0] - 2, -1, -1):
        r = r + part[b]
    assert not torch.equal(_bits(r), _bits(s)), "%s: reverse slot order gives the same bits - the check has no teeth" % tag


# ---- weight gradient ---------------------------------------------------------------------------------------------------
REF_CASES = [("ref_s1", 32, 64, 1, 2, 37, 300, {}, None, None), ("ref_s2", 64, 128, 2, 2, 37, 301, {}, None, None),
             ("ref_narrow", 40, 20, 1, 3, 19, 45, {}, None, None)]


@pytest.mark.parametrize("c", [pytest.param(c, id=c[0]) for c in WGRAD_CASES + REF_CASES])
def test_wgrad_ordered(cuda, knobs, capfd, c):
    from adaptivepnp_sci_b200 import engine
    cid, Cin, Cout, stride, N, H, W, env, prefix = c[:9]
    for k, v in env.items():
        knobs.setenv(k, v)
    impl_ = 1 if cid.startswith("ref") else 0
    g = torch.Generator().manual_seed(Cin * 7 + Cout + stride + 1)
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    q = (lambda t: t) if impl_ else tf32
    x = q(torch.randn(N, H, W, Cin, generator=g)).to(cuda)
    dz = q(torch.randn(N, Ho, Wo, Cout, generator=g)).to(cuda)
    osc = (0.5 + torch.rand(Cout, generator=g)).to(cuda)
    dw0 = torch.randn(9, Cout, Cin, generator=g).to(cuda)                  # the gradient is ACCUMULATED onto this
    n = 9 * Cout * Cin
    d = engine.WgradDesc(x.data_ptr(), dz.data_ptr(), osc.data_ptr(), dw0.data_ptr(), N, H, W, Cin, Cout, stride)
    need = _L().lib.sci_conv3x3_wgrad_workspace_bytes(ctypes.byref(d), impl_)
    slots = need // (4 * n)
    assert need == 4 * n * slots
    tiles = N * -(-Ho // 8) * -(-Wo // 8)
    if not impl_:
        swap = Cout < Cin or (Cin == 32 and Cout == 32)
        want = min(tiles, 148) if prefix == "wgrad v3" else max(1, min(tiles, 148 // (3 * (1 if swap else -(-Cout // 128)))))
        assert slots == want
    ws = torch.empty(need // 4, dtype=torch.float32, device=cuda)
    d.workspace, d.workspace_bytes = ws.data_ptr(), need
    runs = []
    capfd.readouterr()
    for _ in range(2):
        dw = dw0.clone()
        d.dw = dw.data_ptr()
        ws.fill_(float("nan"))
        _L().check(_L().lib.sci_conv3x3_wgrad(ctypes.byref(d), impl_, _L().stream()), "sci_conv3x3_wgrad")
        torch.cuda.synchronize()
        runs.append((dw, ws.view(slots, n).clone()))
    if prefix:
        assert prefix + " plan:" in capfd.readouterr().err
    (dw, part), (dw2, part2) = runs
    _check_slots(cid, part, dw0.reshape(-1), dw.reshape(-1))
    assert torch.equal(_bits(dw), _bits(dw2)) and torch.equal(_bits(part), _bits(part2)), "two calls differ"
    # float64, with the bound of the atomic form (same chain: CTA accumulator, one add per slot, the start value)
    xp = F.pad(x.double(), (0, 0, 1, 1, 1, 1))
    dz64 = dz.double().reshape(-1, Cout)
    sums, S = [], []
    for r in range(3):
        for s in range(3):
            xs = xp[:, r:r + stride * (Ho - 1) + 1:stride, s:s + stride * (Wo - 1) + 1:stride].reshape(-1, Cin)
            sums.append(dz64.t() @ xs)
            S.append(dz64.abs().t() @ xs.abs())
    gsum, S = torch.stack(sums), torch.stack(S)
    o64 = osc.double()[None, :, None]
    ref = dw0.double() + o64 * gsum
    inner = 8 + 8 * -(-tiles // slots) if not impl_ else -(-N * Ho * Wo // slots) + 16 + 1     # + 1: fp32 product rounding
    eb = o64 * C_ACC * (inner + slots + 1) * 2.0 ** -24 * S + 2.0 ** -23 * ((o64 * gsum).abs() + ref.abs())
    err = (dw.double() - ref).abs()
    assert bool((err <= eb).all()), "%s: max err/bound %g" % (cid, float((err / eb).max()))


# ---- column sums fused into the data gradient ----------------------------------------------------------------------------
COLSUM_CASES = [
    # id, Cin, Cout, pixel_shuffle, residual, mask_relu, col_s2, H, W (of the GEMM: the stored output is 2H x 2W with ps)
    ("relu_s1", 64, 64, 0, False, 1, False, 37, 300),
    ("relu_s12_res", 64, 64, 0, True, 1, True, 37, 300),
    ("norelu_s12", 32, 32, 0, False, 0, True, 37, 300),
    ("ps128_res", 64, 128, 1, True, 1, True, 19, 151),
    ("ps256_two_launches", 128, 256, 1, False, 1, True, 19, 151),
]


@pytest.mark.parametrize("c", [pytest.param(c, id=c[0]) for c in COLSUM_CASES])
def test_fused_column_sums_ordered(cuda, knobs, capfd, c):
    from adaptivepnp_sci_b200 import engine
    cid, Cin, Cout, ps, res, mrelu, want_s2, H, W = c
    N = 2
    g = torch.Generator().manual_seed(Cin + 3 * Cout + ps)
    Cq, oh, ow = (Cout // 4, 2 * H, 2 * W) if ps else (Cout, H, W)
    x = tf32(torch.randn(N, H, W, Cin, generator=g)).to(cuda)
    w = tf32(0.2 * torch.randn(9, Cout, Cin, generator=g)).to(cuda)
    r = torch.randn(N, oh, ow, Cq, generator=g).to(cuda) if res else None
    mask = torch.randn(N, oh, ow, Cq, generator=g).to(cuda)
    mask[torch.rand(mask.shape, generator=g).to(cuda) < 0.25] = 0.0
    s1_0 = torch.full((Cq,), 0.25, device=cuda)
    s2_0 = torch.full((Cq,), -0.5, device=cuda)

    def run(ws):
        y = torch.full((N, oh, ow, Cq), float("nan"), device=cuda)
        s1, s2 = s1_0.clone(), (s2_0.clone() if want_s2 else None)
        d = engine.ConvDesc()
        for k, v in dict(x=x, w=w, residual=r, y=y, N=N, H=H, W=W, Cin=Cin, Cout=Cout, stride=1, pixel_shuffle=ps,
                         round_tf32=1, mask_y=mask, col_s1=s1, col_s2=s2, mask_relu=mrelu).items():
            setattr(d, k, v.data_ptr() if isinstance(v, torch.Tensor) else v)
        need = _L().lib.sci_conv3x3_fwd_workspace_bytes(ctypes.byref(d), 0)
        if ws is not None:
            ws.fill_(float("nan"))
            d.workspace, d.workspace_bytes = ws.data_ptr(), need
        _L().check(_L().lib.sci_conv3x3_dgrad(ctypes.byref(d), 0, _L().stream()), "sci_conv3x3_dgrad")
        torch.cuda.synchronize()
        return need, y, s1, s2

    capfd.readouterr()
    need, ya, s1a, s2a = run(None)
    assert "mode 4" in capfd.readouterr().err
    assert need > 0 and need % (8 * Cq) == 0
    slots = need // (8 * Cq)
    ws = torch.empty(need // 4, dtype=torch.float32, device=cuda)
    _, y, s1, s2 = run(ws)
    part = ws.view(slots, 2, Cq).clone()
    plans = capfd.readouterr().err
    assert "mode 5" in plans and "mode 4" not in plans
    _, y2, s1b, s2b = run(ws)
    assert torch.equal(_bits(y), _bits(ya)), "dz differs from the atomic form's"
    assert torch.equal(_bits(y), _bits(y2)) and torch.equal(_bits(s1), _bits(s1b)), "two calls differ"
    _check_slots(cid + " s1", part[:, 0], s1_0, s1)
    if want_s2:
        assert torch.equal(_bits(s2), _bits(s2b))
        _check_slots(cid + " s2", part[:, 1], s2_0, s2)
    # float64: the sums of exactly the stored dz (the bound of the atomic form: lane column sum, the units of the CTA, one
    # add per slot, the start value; col_s2 adds the rounding of each product)
    n_pix = N * oh * ow
    depth = 32 + (n_pix + 31) // 32 + slots + 1
    for got, start, wgt in ((s1, 0.25, None), (s2, -0.5, mask.double())):
        if got is None:
            continue
        own = (y.double() if wgt is None else y.double() * wgt).reshape(-1, Cq)
        b = C_ACC * depth * 2.0 ** -24 * (own.abs().sum(0) + abs(start)) + (0 if wgt is None else 2.0 ** -24 * own.abs().sum(0))
        e = (got.double() - (start + own.sum(0))).abs()
        assert bool((e <= b).all()), "%s: column sums max err/bound %g" % (cid, float((e / b).max()))
    for got, ref in ((s1, s1a), (s2, s2a)):                       # ordered and atomic sums agree to rounding
        if got is not None:
            assert float((got - ref).abs().max()) <= 1e-4 * float(ref.abs().max() + 1)


# ---- act_bwd -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C,relu,y_null,want_s2,n_pix", [(48, 1, False, True, 22200), (64, 0, False, True, 2 * 37 * 300),
                                                         (96, 1, False, False, 12345), (256, 1, False, True, 3001),
                                                         (32, 0, True, False, 777)])
def test_act_bwd_ordered(cuda, C, relu, y_null, want_s2, n_pix):
    g = torch.Generator().manual_seed(C * 31 + n_pix)
    dy = torch.randn(n_pix, C, generator=g).to(cuda)
    y = None if y_null else torch.randn(n_pix, C, generator=g).to(cuda)
    if y is not None:
        y[torch.rand(y.shape, generator=g).to(cuda) < 0.2] = 0.0
    rows = max(1, 256 // C)
    grid = min(148 * 8, -(-n_pix // rows))
    nb = _L().lib.sci_act_bwd_workspace_bytes(n_pix, C)
    assert nb == grid * 2 * C * 4
    ws = torch.empty(nb // 4, dtype=torch.float32, device=cuda)
    s1_0, s2_0 = torch.full((C,), 0.25, device=cuda), torch.full((C,), -0.5, device=cuda)
    p = _L().ptr
    dza = dy.clone()
    s1a, s2a = s1_0.clone(), s2_0.clone()
    _L().call("sci_act_bwd", p(dy), p(y), p(dza), n_pix, C, relu, p(s1a), p(s2a) if want_s2 else None, _L().stream())
    runs = []
    for _ in range(2):
        dz = torch.full_like(dy, float("nan"))
        s1, s2 = s1_0.clone(), s2_0.clone()
        ws.fill_(float("nan"))
        _L().call("sci_act_bwd_ordered", p(dy), p(y), p(dz), n_pix, C, relu, p(s1), p(s2) if want_s2 else None, p(ws), nb,
                  _L().stream())
        torch.cuda.synchronize()
        runs.append((dz, s1, s2, ws.view(grid, 2, C).clone()))
    (dz, s1, s2, part), (dz2, s1b, s2b, _) = runs
    assert torch.equal(_bits(dz), _bits(dza)), "dz differs from sci_act_bwd's"
    assert torch.equal(_bits(dz), _bits(dz2)) and torch.equal(_bits(s1), _bits(s1b)) and torch.equal(_bits(s2), _bits(s2b))
    _check_slots("act_bwd s1", part[:, 0], s1_0, s1)
    if want_s2:
        _check_slots("act_bwd s2", part[:, 1], s2_0, s2)
    else:
        assert torch.equal(s2, s2_0)
    # float64 bound of the atomic form: each thread's grid-stride chain, the block's row combine, one add per slot, start
    depth = -(-n_pix // (grid * rows)) + rows + grid + 1
    y64 = torch.zeros_like(dz, dtype=torch.float64) if y is None else y.double()
    for got, start, t in ((s1, 0.25, dz.double()), (s2, -0.5, dz.double() * y64)):
        if got is s2 and not want_s2:
            continue
        b = C_ACC * (depth + 1) * 2.0 ** -24 * (t.abs().sum(0) + abs(start))
        e = (got.double() - (start + t.sum(0))).abs()
        assert bool((e <= b).all()), "act_bwd: max err/bound %g" % float((e / b).max())


# ---- engines: one fine-tune call twice -----------------------------------------------------------------------------------
def _ffdnet_gray(cuda):
    from adaptivepnp_sci_b200.network_ffdnet import FFDNet
    m = FFDNet(1, 1, 64, 15, 'R')
    m.load_state_dict(torch.load(os.path.join(ROOT, "model_zoo", "ffdnet_gray.pth")), strict=True)
    return m.eval().cuda()


NETS = {"fastdvd_color": (lambda dev: _fastdvd(dev), 3), "fastdvd_gray": (lambda dev: _gray_model(dev), 1),
        "ffdnet_color": (lambda dev: _ffdnet(dev), 3), "ffdnet_gray": (_ffdnet_gray, 1)}


@pytest.mark.parametrize("net", list(NETS))
def test_engine_finetune_bit_identical(cuda, impl, net):
    from adaptivepnp_sci_b200 import fastdvdnet_adapter, ffdnet_adapter
    make, C = NETS[net]
    B, H, W = 7, 36, 44                          # ragged: 7 frames, sizes that fill no tile of the kernels
    g = torch.Generator().manual_seed(11)
    v = torch.rand(B, C, H, W, generator=g).to(cuda)
    phi = (torch.rand(B, H, W, generator=g) > 0.5).float().to(cuda)
    y = (phi * v.mean(1)).sum(0).contiguous()
    noise = np.random.RandomState(5).standard_normal((B, C, H, W)) * (10 / 255)
    runs = []
    for _ in range(2):
        m = make(cuda)
        sd0 = {k: t.clone() for k, t in m.state_dict().items()}
        if net.startswith("fastdvd"):
            out = fastdvdnet_adapter.finetune_and_denoise(v, phi, y, 12 / 255, m, [2e-4, 1e-4], [2, 1], noise=noise)
            eng = fastdvdnet_adapter._unwrap(m).engine()
        else:
            out = ffdnet_adapter.finetune_and_denoise(v, phi, y, 25 / 255, m, 2e-4, 2)
            eng = ffdnet_adapter._unwrap(m).engine()
        torch.cuda.synchronize()
        sd = {k: t.clone() for k, t in m.state_dict().items()}
        assert max(float((sd[k].float() - sd0[k].float()).abs().max()) for k in sd) > 1e-6, "the fine-tune did not move"
        runs.append((out.clone(), sd, eng.bucket.exp_avg.clone(), eng.bucket.exp_avg_sq.clone(), eng.bucket.grad.clone()))
    (o1, sd1, m1, v1, g1), (o2, sd2, m2, v2, g2) = runs
    assert float(g1.abs().max()) > 0
    for k in sd1:
        if sd1[k].dtype == torch.float32:
            assert torch.equal(_bits(sd1[k]), _bits(sd2[k])), "weights differ: " + k
        else:
            assert torch.equal(sd1[k], sd2[k])
    for a, b, what in ((m1, m2, "exp_avg"), (v1, v2, "exp_avg_sq"), (g1, g2, "grad"), (o1, o2, "output")):
        assert torch.equal(_bits(a), _bits(b)), what + " differs"


# ---- public entry points ------------------------------------------------------------------------------------------------
def _same_result(r1, r2, m1, m2, n_img):
    u8 = lambda a: np.ascontiguousarray(a).view(np.uint8)
    for i in range(n_img):
        assert r1[i].shape == r2[i].shape and np.array_equal(u8(r1[i]), u8(r2[i])), "output %d differs" % i
    for i in (2, 4):                                          # PSNR lists (fp64 diagnostics, atomics, never fed back)
        a, b = np.array(r1[i], dtype=np.float64), np.array(r2[i], dtype=np.float64)
        assert a.shape == b.shape and np.all(np.abs(a - b) <= 1e-12 * np.abs(a))
    s1, s2 = m1.state_dict(), m2.state_dict()
    for k in s1:
        assert torch.equal(s1[k].reshape(-1).view(torch.uint8), s2[k].reshape(-1).view(torch.uint8)), k


@pytest.mark.parametrize("den", ["fastdvd_color", "ffdnet_color"])
def test_two_stage_bayer_bit_identical(cuda, den):
    from adaptivepnp_sci_b200.dvp_linear_inv_2_stage_ADMM_tensor_online import np2tch_cuda, twoStageAdmm_denoise_bayer
    from adaptivepnp_sci_b200.utilspy import worker_init_fn
    from oracle import synthetic
    d = np.load(os.path.join(G, "loops.npz"))
    meas, mask, orig = synthetic.make_case(64, 64, 8, 3000, bayer=True)
    rs, ms = [], []
    for _ in range(2):
        m = _fastdvd(cuda) if den == "fastdvd_color" else _ffdnet(cuda)
        worker_init_fn(0)
        sig = [12 / 255, 6 / 255] if den == "fastdvd_color" else [25 / 255, 12 / 255]
        r = twoStageAdmm_denoise_bayer(meas, mask, 1, 0.01, den, [4, 3], False, sig, x0_bayer=np2tch_cuda(d["s2_warm"]),
                                       X_orig=orig, model_denoise=m, model_demosaic=None, show_iqa=True,
                                       demosaic_method='malvar2004', lr_=2e-6, interval_iter=3, logf=io.StringIO(),
                                       update_=True, update_per_iter=2, update_times=-1)
        rs.append(r)
        ms.append(m)
    _same_result(rs[0], rs[1], ms[0], ms[1], 2)


def test_two_stage_gray_fastdvd_bit_identical(cuda):
    from adaptivepnp_sci_b200.dvp_linear_inv_2_stage_ADMM_tensor_online import twoStageAdmm_denoise_gray
    from adaptivepnp_sci_b200.utilspy import worker_init_fn
    from oracle import synthetic
    meas, mask, orig = synthetic.make_case(64, 64, 8, 1001, bayer=False)
    warm = np.clip(meas[:, :, None] * mask / np.maximum(mask.sum(2, keepdims=True), 1), 0, 1).astype(np.float32)
    rs, ms = [], []
    for _ in range(2):
        m = _gray_model(cuda)
        worker_init_fn(0)
        r = twoStageAdmm_denoise_gray(meas, mask, 'fastdvd_gray', iter_max=[4, 3], sigma=[12 / 255, 6 / 255],
                                      x0=torch.from_numpy(warm).cuda(), X_orig=orig, model_denoise=m, logf=io.StringIO(),
                                      lr_=2e-6, interval_iter=3, update_=True, update_per_iter=2)
        rs.append(r)
        ms.append(m)
    _same_result(rs[0], rs[1], ms[0], ms[1], 2)


# ---- two processes over gloo ---------------------------------------------------------------------------------------------
TH, TW, TB = 352, 32, 3          # two strips of 176 rows (as tests/test_gpu_tiled.py)
SH, SW, SB = 64, 64, 8


def _worker(rank, world, port, q, mode):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK="0", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port),
                      SCI_CONV_IMPL="tc")
    from adaptivepnp_sci_b200 import parallel
    from adaptivepnp_sci_b200.dvp_linear_inv_2_stage_ADMM_tensor_online import twoStageAdmm_denoise_bayer
    from adaptivepnp_sci_b200.utilspy import worker_init_fn
    from adaptivepnp_sci_b200.synthetic import make_case
    ctx = parallel.init(backend="gloo")
    kw = dict(show_iqa=True, demosaic_method='malvar2004', lr_=2e-6, update_=True, logf=io.StringIO(), update_times=-1)
    m = _fastdvd(None)
    if mode == "tiled":
        tile = parallel.TileContext(ctx, TH, TW)
        meas, mask, orig = make_case(TH, TW, TB, 77, bayer=True)
        warm = np.clip(meas[:, :, None] * mask / np.maximum(mask.sum(2, keepdims=True), 1), 0, 1).astype(np.float32)
        worker_init_fn(0)
        r = twoStageAdmm_denoise_bayer(tile.slice_rows(meas), tile.slice_rows(mask), 1, 0.01, 'fastdvd_color', [4], False,
                                       [12 / 255], x0_bayer=torch.from_numpy(tile.slice_rows(warm)).cuda(),
                                       X_orig=tile.slice_rows(orig), model_denoise=m, tile=tile, interval_iter=2,
                                       update_per_iter=1, **kw)
    else:
        meas, mask, orig = make_case(SH, SW, SB, 3000 + rank, bayer=True)
        warm = np.clip(meas[:, :, None] * mask / np.maximum(mask.sum(2, keepdims=True), 1), 0, 1).astype(np.float32)
        worker_init_fn(0)
        r = twoStageAdmm_denoise_bayer(meas, mask, 1, 0.01, 'fastdvd_color', [4], False, [12 / 255],
                                       x0_bayer=torch.from_numpy(warm).cuda(), X_orig=orig, model_denoise=m,
                                       grad_sync=ctx.grad_sync, interval_iter=2, update_per_iter=2, **kw)
    q.put((rank, r[0], r[1], {k: t.cpu().numpy() for k, t in m.state_dict().items()}))
    ctx.finalize()


def _two_ranks(mode):
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctxm = mp.get_context("spawn")
    q = ctxm.Queue()
    procs = [ctxm.Process(target=_worker, args=(r, 2, port, q, mode)) for r in range(2)]
    for p in procs:
        p.start()
    outs = sorted((q.get(timeout=600) for _ in range(2)), key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return outs


@pytest.mark.parametrize("mode", ["tiled", "shared"])
def test_two_processes_bit_identical(cuda, mode):
    a, b = _two_ranks(mode), _two_ranks(mode)
    for (ra, rgb_a, x_a, sd_a), (rb, rgb_b, x_b, sd_b) in zip(a, b):
        assert ra == rb
        u8 = lambda t: np.ascontiguousarray(t).view(np.uint8)
        assert np.array_equal(u8(rgb_a), u8(rgb_b)) and np.array_equal(u8(x_a), u8(x_b))
        for k in sd_a:
            assert np.array_equal(u8(sd_a[k]), u8(sd_b[k])), k
    if mode == "shared":                                           # one shared set of weights on both ranks
        for k in a[0][3]:
            assert np.array_equal(np.ascontiguousarray(a[0][3][k]).view(np.uint8), np.ascontiguousarray(a[1][3][k]).view(np.uint8)), k
