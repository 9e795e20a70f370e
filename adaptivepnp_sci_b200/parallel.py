"""Single-node multi-GPU plumbing: one process per GPU (torchrun), NCCL over NVLink only where the path
really exchanges data.

* Measurement groups / videos are independent work units (SURVEY §8(e)): ``my_units`` deals them round-robin to
  the ranks, ``gather_units`` collects the numpy results on rank 0 (object gather; no collective touches the
  per-iteration data path).
* Shared-weight online fine-tuning (BASELINE config 4): every rank fine-tunes the SAME denoiser weights on its
  own group; ``grad_sync`` all-reduces (mean) the flat gradient bucket — one NCCL call of <= 10 MB per Adam step —
  so all ranks take identical steps.  This is a semantic change against the reference (which fine-tunes
  sequentially, group after group, ``reuse_model=True``) and is only used when requested.

On CPU (``gloo``) the same code paths run in the unit tests (tests/test_parallel_cpu.py).
"""
import os

import torch


class Context:
    def __init__(self, rank, world, local_rank, backend):
        self.rank, self.world, self.local_rank, self.backend = rank, world, local_rank, backend

    def my_units(self, n):
        """Indices of the independent units (measurement groups) this rank owns."""
        return list(range(self.rank, n, self.world))

    def check_even_split(self, n, what="units"):
        """Lock-step collectives (the shared-weight gradient all-reduce) need every rank to own the same number of units:
        a rank without a unit would never enter the all-reduce and the others would hang in NCCL until the timeout."""
        if n % self.world != 0:
            raise ValueError("%d %s do not divide evenly over %d ranks: a shared-weight run needs equal shares "
                             "(every rank joins every gradient all-reduce)" % (n, what, self.world))

    def gather_units(self, results):
        """dict{unit: payload} from every rank -> merged dict on rank 0 (others get {})."""
        if self.world == 1:
            return results
        import torch.distributed as dist
        out = [None] * self.world if self.rank == 0 else None
        dist.gather_object(results, out, dst=0)
        merged = {}
        if self.rank == 0:
            for d in out:
                merged.update(d)
        return merged

    def grad_sync(self, flat_grad):
        """Mean all-reduce of the flat gradient bucket (identity on one rank)."""
        if self.world > 1:
            import torch.distributed as dist
            if self.backend == "nccl":
                dist.all_reduce(flat_grad, op=dist.ReduceOp.AVG)
            else:
                dist.all_reduce(flat_grad, op=dist.ReduceOp.SUM)
                flat_grad.div_(self.world)
        return flat_grad

    def broadcast_(self, tensor, src=0):
        if self.world > 1:
            import torch.distributed as dist
            dist.broadcast(tensor, src)
        return tensor

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()

    def finalize(self):
        if self.world > 1:
            import torch.distributed as dist
            if dist.is_initialized():
                dist.destroy_process_group()


class P2PRegion:
    """One cudaMalloc'ed region per rank, mapped into its two neighbours through CUDA IPC (``sci_p2p_*``):

        [ flags: u32 from_up @0, u32 from_down @4 ... 256 B ][ slot(parity 0, TOP) | slot(0, BOTTOM) | slot(1, TOP) | slot(1, BOTTOM) ]

    ``exchange`` stores this rank's boundary rows straight into the neighbours' slots over NVLink (``sci_halo_send``) and
    assembles its halo-extended strip from its own slots once the neighbours' sequence numbers have arrived
    (``sci_halo_assemble``): no NCCL call, no staging copy, no host synchronisation.  All ranks count exchanges in lock-step."""
    HDR = 256

    def __init__(self, ctx, slot_bytes):
        import ctypes
        import torch.distributed as dist
        from ._lib import call
        self.ctx, self.slot = ctx, (int(slot_bytes) + 255) // 256 * 256
        self.seq = 0
        base = ctypes.c_void_p()
        call("sci_p2p_alloc", self.HDR + 4 * self.slot, ctypes.byref(base))
        self.base = base.value
        h = ctypes.create_string_buffer(64)
        call("sci_p2p_get_handle", ctypes.c_void_p(self.base), h)
        handles = [None] * ctx.world
        dist.all_gather_object(handles, bytes(h.raw))
        self.peer = {}
        for r in (ctx.rank - 1, ctx.rank + 1):
            if 0 <= r < ctx.world:
                q = ctypes.c_void_p()
                call("sci_p2p_open_handle", ctypes.create_string_buffer(handles[r], 64), ctypes.byref(q))
                self.peer[r] = q.value
        dev = torch.device("cuda", torch.cuda.current_device())
        self.scratch = torch.zeros(2, dtype=torch.int32, device=dev)          # [done counter of the send kernel, error word]
        dist.barrier()                                                        # every region is mapped before anyone stores into it

    def slot_ptr(self, base, parity, side):
        return base + self.HDR + (parity * 2 + side) * self.slot

    def exchange(self, own, top, bot, halo):
        import ctypes
        from ._lib import call, ptr, stream
        B, C, rows, W = own.shape
        if B * C * halo * W * 4 > self.slot:
            raise ValueError("halo of %d bytes exceeds the P2P slot (%d)" % (B * C * halo * W * 4, self.slot))
        self.seq += 1
        par, r = self.seq & 1, self.ctx.rank
        vp = ctypes.c_void_p
        up, down = self.peer.get(r - 1) if top else None, self.peer.get(r + 1) if bot else None
        # my top rows are the BOTTOM halo (side 1, flag from_down @4) of the upper neighbour, and vice versa
        call("sci_halo_send", ptr(own), B * C, rows, W, halo,
             vp(self.slot_ptr(up, par, 1)) if up else None, vp(self.slot_ptr(down, par, 0)) if down else None,
             vp(up + 4) if up else None, vp(down) if down else None, self.seq, vp(self.scratch.data_ptr()), stream())
        ext = torch.empty((B, C, top + rows + bot, W), dtype=own.dtype, device=own.device)
        call("sci_halo_assemble", ptr(own), B * C, rows, W, top, bot, vp(self.slot_ptr(self.base, par, 0)),
             vp(self.slot_ptr(self.base, par, 1)), vp(self.base), vp(self.base + 4), self.seq, ptr(ext),
             vp(self.scratch.data_ptr() + 4), stream())
        return ext

    def send_tv(self, x, b, c_b, top, bot):
        """The TV prior's halo: f = x + c_b*b of this strip's first / last 8 rows goes straight into the neighbours' slots
        (``sci_halo_send_tv``).  Returns what ``sci_tv_strip_main`` needs to read this rank's own slots in place: (halo_top,
        halo_bot, flag_top, flag_bot, seq, err) as raw addresses (None where there is no neighbour).  The slots of this
        exchange are read again by the fix-up pass (``sci_tv_strip_finish``); the next exchange is issued after it in stream
        order, which keeps the parity argument of the class docstring."""
        from . import ops
        B, rows, W = x.shape
        if B * ops.TV_HALO * W * 4 > self.slot:
            raise ValueError("TV halo of %d bytes exceeds the P2P slot (%d)" % (B * ops.TV_HALO * W * 4, self.slot))
        self.seq += 1
        par, r = self.seq & 1, self.ctx.rank
        up, down = self.peer.get(r - 1) if top else None, self.peer.get(r + 1) if bot else None
        ops.halo_send_tv(x, b, c_b, self.slot_ptr(up, par, 1) if up else None, self.slot_ptr(down, par, 0) if down else None,
                         up + 4 if up else None, down if down else None, self.seq, self.scratch.data_ptr())
        return (self.slot_ptr(self.base, par, 0) if top else None, self.slot_ptr(self.base, par, 1) if bot else None,
                self.base if top else None, self.base + 4 if bot else None, self.seq, self.scratch.data_ptr() + 4)

    def check(self):
        """Host-side check of the bounded wait (call at a synchronisation point)."""
        e = int(self.scratch[1])
        if e:
            raise RuntimeError("P2P halo exchange: neighbour %s did not deliver within 10 s" % ("above" if e == 1 else "below"))

    def close(self):
        """Collective (every rank closes its region at the same point, like ``enable_p2p``): a neighbour's stream may still hold
        stores into this region, so all devices drain and all ranks meet before anything is unmapped or freed."""
        from ._lib import call
        import ctypes
        import torch.distributed as dist
        torch.cuda.synchronize()
        if self.ctx.world > 1 and dist.is_initialized():
            dist.barrier()
        for q in self.peer.values():
            call("sci_p2p_close_handle", ctypes.c_void_p(q))
        self.peer = {}
        if self.base:
            call("sci_p2p_free", ctypes.c_void_p(self.base))
            self.base = None


class TileContext:
    """Row-strip spatial tiling of ONE large frame over the ranks (BASELINE config 5, SURVEY 8(e)).

    Rank r owns the contiguous rows [r*rows, (r+1)*rows) of every plane (rows % 4 == 0 keeps the Bayer phase, the
    stride-2 and the PixelShuffle phases aligned).  Pixel-wise kernels (projection, dual updates) need nothing from
    the neighbours; stencils do:

    * Malvar demosaic: 2 rows of the merged mosaic,
    * denoiser: ``halo`` rows of its RGB input (FastDVDnet two-stage cascade: receptive field -77..+73 rows -> 80;
      FFDNet-colour: -24..+25 -> 28), exchanged once per ADMM iteration; the strip is then denoised with its halo and
      cropped ("overlap-tile"), so zero padding is only ever applied at true image borders.

    * TV prior (``tv_chambolle``): 8 rows of f = x + c_b*b, exchanged once per call (the kernel runs all inner iterations
      on chip, and a pixel depends only on rows within +-8).

    ``exchange`` moves the halo rows peer to peer: after ``enable_p2p`` the boundary rows are stored straight into the
    neighbour's memory over NVLink by ``sci_halo_send`` / ``sci_halo_assemble`` (``P2PRegion``); without it (CPU tests,
    ``SCI_TILE_P2P=0``) with point-to-point sends of torch.distributed.  The only collective on the per-iteration path is
    the TV prior's all-gather of its early-stop energies (``world`` x 4B x 8 doubles per call, in-stream on NCCL); the
    other reductions are the scalar PSNR sums, the fine-tune loss/gradient all-reduce (SUM: the loss is normalised by the
    pixel count of the whole frame) and the final gather of the result strips."""

    def __init__(self, ctx, H_total, W):
        if H_total % (4 * ctx.world) != 0:
            raise ValueError("tiled mode needs H divisible by 4*world_size (got H=%d, world=%d)" % (H_total, ctx.world))
        self.ctx = ctx
        self.rank, self.world = ctx.rank, ctx.world
        self.H_total, self.W = H_total, W
        self.rows = H_total // ctx.world
        self.r0 = self.rank * self.rows
        self.total_pixels = H_total * W
        self.p2p = None
        self.halo_bytes_moved = 0
        # results: True = only rank 0 assembles (and copies to the host) the full-frame outputs, the other ranks get None
        # for the two image arrays - what a job that writes ONE result file needs; False = every rank gets the full frame
        self.gather_root_only = False

    def enable_p2p(self, max_planes, max_halo):
        """Peer-to-peer halo exchange over NVLink (``P2PRegion``) for CUDA strips of fp32 planes; every rank must call it with
        the same sizes.  ``SCI_TILE_P2P=0`` keeps the point-to-point sends of torch.distributed (NCCL / gloo)."""
        if self.world == 1 or not torch.cuda.is_available() or os.environ.get("SCI_TILE_P2P", "1") == "0":
            return False
        need = max_planes * max_halo * self.W * 4
        if self.p2p is None or self.p2p.slot < need:
            if self.p2p is not None:
                self.p2p.close()
            self.p2p = P2PRegion(self.ctx, need)
        return True

    def slice_rows(self, a):
        """numpy/torch [H_total, ...] -> this rank's rows."""
        return a[self.r0:self.r0 + self.rows]

    def halo_sizes(self, halo):
        if self.world > 1 and halo > self.rows:
            # a strip shorter than the denoiser's receptive field would need rows from rank +-2 as well; clamping the halo
            # would silently break the "tiled == un-tiled" guarantee
            raise ValueError("tiled mode: strips of %d rows are shorter than the %d-row halo the denoiser needs "
                             "(use fewer ranks for a %d-row frame)" % (self.rows, halo, self.H_total))
        return (halo if self.rank > 0 else 0), (halo if self.rank < self.world - 1 else 0)

    def exchange(self, own, halo):
        """own [B,C,rows,W] (contiguous, this rank's rows) -> (ext [B,C,top+rows+bot,W], top)."""
        top, bot = self.halo_sizes(halo)
        B, C, rows, W = own.shape
        self.halo_bytes_moved += (top + bot) * B * C * W * own.element_size()
        if self.world > 1 and self.p2p is not None and own.is_cuda and own.dtype == torch.float32 and W % 4 == 0:
            return self.p2p.exchange(own.contiguous(), top, bot, halo), top
        ext = torch.empty((B, C, top + rows + bot, W), dtype=own.dtype, device=own.device)
        ext[:, :, top:top + rows].copy_(own)
        if self.world == 1:
            return ext, 0
        rcv_top, rcv_bot = self._sendrecv_rows(own, top, bot)
        if rcv_top is not None:
            ext[:, :, :top].copy_(rcv_top)
        if rcv_bot is not None:
            ext[:, :, top + rows:].copy_(rcv_bot)
        return ext, top

    def _sendrecv_rows(self, own, top, bot):
        """Point-to-point sends of torch.distributed: my first ``top`` rows up and last ``bot`` rows down; returns the rows
        received from the upper / lower neighbour (None where there is none)."""
        import torch.distributed as dist
        rows = own.shape[-2]
        host = self.ctx.backend != "nccl"          # gloo moves CUDA halos through host memory (tests / CPU runs)
        ops, bufs = [], {}
        if top:      # upper neighbour: send my first rows, receive its last rows
            snd = own[..., :top, :].contiguous()
            snd = snd.cpu() if host else snd
            rcv = torch.empty_like(snd)
            ops += [dist.P2POp(dist.isend, snd, self.rank - 1), dist.P2POp(dist.irecv, rcv, self.rank - 1)]
            bufs["top"] = (rcv, snd)
        if bot:
            snd = own[..., rows - bot:, :].contiguous()
            snd = snd.cpu() if host else snd
            rcv = torch.empty_like(snd)
            ops += [dist.P2POp(dist.isend, snd, self.rank + 1), dist.P2POp(dist.irecv, rcv, self.rank + 1)]
            bufs["bot"] = (rcv, snd)
        for w in dist.batch_isend_irecv(ops):
            w.wait()
        got = {k: v[0].to(own.device) for k, v in bufs.items()}
        return got.get("top"), got.get("bot")

    def tv_chambolle(self, x, b, c_b, theta, b_out, s_b, clip, ws, weight=0.1, eps=2.0e-4, n_iter_max=5, nstop_out=None):
        """``ops.tv_chambolle`` on this rank's strip x [B, rows, W] (``ws``: ``ops.TvStripWorkspace``).  Halo of 8 rows of
        f = x + c_b*b from each neighbour (peer to peer after ``enable_p2p``, else torch.distributed), main pass, all-gather
        of the early-stop energies, decision + fix-up pass.  Every rank sums the gathered energies in rank order, so all
        make the same stop decisions; own pixels are those of the un-tiled kernel bit for bit given the same decisions."""
        from . import ops
        B, rows, W = x.shape
        top, bot = self.halo_sizes(ops.TV_HALO)
        kw = dict(weight=weight, eps=eps, n_iter_max=n_iter_max)
        halo_top = halo_bot = None
        wait = {}
        if self.world > 1:
            self.halo_bytes_moved += (top + bot) * B * W * 4
            if self.p2p is not None and x.is_cuda:
                halo_top, halo_bot, ft, fb, seq, err = self.p2p.send_tv(x, b, c_b, top, bot)
                wait = dict(flag_top=ft, flag_bot=fb, seq=seq, err=err)
            else:
                f = x if b is None else ops.axpy(x, c_b, b)
                halo_top, halo_bot = self._sendrecv_rows(f, top, bot)
        esum = ops.tv_strip_main(x, b, c_b, theta, b_out, s_b, clip, ws, self.r0, self.H_total, halo_top, halo_bot,
                                 **kw, **wait)
        esum_all = esum.view(1, *esum.shape)
        if self.world > 1:
            import torch.distributed as dist
            if self.ctx.backend == "nccl":
                esum_all = torch.empty((self.world,) + tuple(esum.shape), dtype=esum.dtype, device=esum.device)
                dist.all_gather_into_tensor(esum_all, esum)
            else:                                   # gloo: through host memory, like gather_rows
                parts = [torch.empty(esum.shape, dtype=esum.dtype) for _ in range(self.world)]
                dist.all_gather(parts, esum.cpu())
                esum_all = torch.stack(parts).to(esum.device)
        return ops.tv_strip_finish(x, b, c_b, theta, b_out, s_b, clip, ws, self.r0, self.H_total, esum_all, halo_top,
                                   halo_bot, nstop_out=nstop_out, **kw)

    def all_reduce_sum(self, t):
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return t

    def gather_rows(self, strip, root_only=False):
        """strip [..., rows, W] on every rank -> full [..., H_total, W] on every rank (``root_only``: on rank 0, None elsewhere)."""
        if self.p2p is not None:
            self.p2p.check()
        if self.world == 1:
            return strip
        import torch.distributed as dist
        src = strip.contiguous()
        if self.ctx.backend != "nccl":
            src = src.cpu()
        if root_only:
            parts = [torch.empty_like(src) for _ in range(self.world)] if self.rank == 0 else None
            dist.gather(src, parts, dst=0)
            return torch.cat(parts, dim=-2).to(strip.device) if self.rank == 0 else None
        parts = [torch.empty_like(src) for _ in range(self.world)]
        dist.all_gather(parts, src)
        return torch.cat(parts, dim=-2).to(strip.device)


def init(backend=None):
    """Reads RANK / LOCAL_RANK / WORLD_SIZE / MASTER_* (torchrun) and initialises the process group."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if backend is None:
        backend = "nccl" if torch.cuda.is_available() else "gloo"
    if torch.cuda.is_available():
        torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        if not dist.is_initialized():
            kw = {}
            if backend == "nccl":
                kw["device_id"] = torch.device("cuda", local_rank)
            dist.init_process_group(backend, **kw)
    return Context(rank, world, local_rank, backend)
