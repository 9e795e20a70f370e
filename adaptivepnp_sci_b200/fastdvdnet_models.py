"""FastDVDnet as used by the reference: ``packages/fastdvdnet/models.py:16-253``.

Parameter containers with the reference's ``state_dict`` key names
(``temp1.inc.convblock.0.weight`` ...), so a ``model.pth`` trained with the public
FastDVDnet code loads unchanged (with or without the ``module.`` prefix of the
``nn.DataParallel`` wrapper the script uses, two_stage_ADMM_Online_FastDVD_Warm.py:240-241).
``forward`` keeps the reference convention (x [N,15,H,W], noise_map [N,1,H,W]) and runs on
the native engine; the hot path calls ``engine.FastDVDnetEngine`` directly on the whole
circular frame sequence so that each temp1 triple is evaluated once.
"""
import torch
import torch.nn as nn


def _cv(ci, co, stride=1, groups=1):
    return nn.Conv2d(ci, co, kernel_size=3, padding=1, stride=stride, groups=groups, bias=False)


class CvBlock(nn.Module):
    def __init__(self, in_ch, out_ch):
        super().__init__()
        self.convblock = nn.Sequential(_cv(in_ch, out_ch), nn.BatchNorm2d(out_ch), nn.ReLU(inplace=True),
                                       _cv(out_ch, out_ch), nn.BatchNorm2d(out_ch), nn.ReLU(inplace=True))


class InputCvBlock(nn.Module):
    def __init__(self, num_in_frames, out_ch, ncolor):
        super().__init__()
        self.interm_ch = 30
        mid = num_in_frames * self.interm_ch
        self.convblock = nn.Sequential(_cv(num_in_frames * (ncolor + 1), mid, groups=num_in_frames), nn.BatchNorm2d(mid),
                                       nn.ReLU(inplace=True), _cv(mid, out_ch), nn.BatchNorm2d(out_ch),
                                       nn.ReLU(inplace=True))


class DownBlock(nn.Module):
    def __init__(self, in_ch, out_ch):
        super().__init__()
        self.convblock = nn.Sequential(_cv(in_ch, out_ch, stride=2), nn.BatchNorm2d(out_ch), nn.ReLU(inplace=True),
                                       CvBlock(out_ch, out_ch))


class UpBlock(nn.Module):
    def __init__(self, in_ch, out_ch):
        super().__init__()
        self.convblock = nn.Sequential(CvBlock(in_ch, in_ch), _cv(in_ch, out_ch * 4), nn.PixelShuffle(2))


class OutputCvBlock(nn.Module):
    def __init__(self, in_ch, out_ch):
        super().__init__()
        self.convblock = nn.Sequential(_cv(in_ch, in_ch), nn.BatchNorm2d(in_ch), nn.ReLU(inplace=True), _cv(in_ch, out_ch))


class DenBlock(nn.Module):
    def __init__(self, num_input_frames=3, num_color_channels=3):
        super().__init__()
        self.chs_lyr0, self.chs_lyr1, self.chs_lyr2 = 32, 64, 128
        self.inc = InputCvBlock(num_input_frames, self.chs_lyr0, num_color_channels)
        self.downc0 = DownBlock(self.chs_lyr0, self.chs_lyr1)
        self.downc1 = DownBlock(self.chs_lyr1, self.chs_lyr2)
        self.upc2 = UpBlock(self.chs_lyr2, self.chs_lyr1)
        self.upc1 = UpBlock(self.chs_lyr1, self.chs_lyr0)
        self.outc = OutputCvBlock(self.chs_lyr0, num_color_channels)
        for m in self.modules():                         # models.py:168-175
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, nonlinearity='relu')

    def conv_specs(self):
        """The 16 convolutions in execution order: (conv, bn or None, relu, stride, pixel_shuffle)."""
        def cvb(b):
            s = b.convblock
            return [(s[0], s[1], True, 1, False), (s[3], s[4], True, 1, False)]
        inc, d0, d1, u2, u1, oc = (self.inc.convblock, self.downc0.convblock, self.downc1.convblock,
                                   self.upc2.convblock, self.upc1.convblock, self.outc.convblock)
        return ([(inc[0], inc[1], True, 1, False), (inc[3], inc[4], True, 1, False)]
                + [(d0[0], d0[1], True, 2, False)] + cvb(d0[3])
                + [(d1[0], d1[1], True, 2, False)] + cvb(d1[3])
                + cvb(u2[0]) + [(u2[1], None, False, 1, True)]
                + cvb(u1[0]) + [(u1[1], None, False, 1, True)]
                + [(oc[0], oc[1], True, 1, False), (oc[3], None, False, 1, False)])


class FastDVDnet(nn.Module):
    """models.py:200-253.  ``num_color_channels=1`` (the grayscale model of ``fastdvdnet_denoiser(gray=True)``,
    test_fastdvdnet.py:149-235) keeps the reference's parameter shapes (``inc`` 3 x (1+1) -> 90 in 3 groups, ``outc``
    32 -> 1) and runs on the colour engine through an exact embedding: a colour-shaped twin holds the same weights with
    zeros in the rows / columns of the two missing colour planes, the frames enter as its first plane, and its first
    output plane is the result - the zero terms add nothing to any accumulator.  The engine takes gray frames [B,1,H,W]
    as they are (its boundary kernels pack them as that first plane and compute only the first output plane).

    Fine-tuning the gray model trains the twin (gradients, ``grad_sync`` and Adam on the twin's flat bucket) and writes the
    result back with ``_restrict_twin``.  The embedded zeros stay exactly +0 through training: their inputs are zero planes
    and the loss never reads output planes 1 and 2, so their gradients are exactly zero, and an Adam step with g = 0 from
    fresh moments m = v = 0 moves nothing."""

    def __init__(self, num_input_frames=5, num_color_channels=3):
        super().__init__()
        if num_input_frames != 5 or num_color_channels not in (1, 3):
            raise NotImplementedError("5-frame models (NUM_IN_FR_EXT = 5) with 3 (colour) or 1 (gray) channels")
        self.num_input_frames = num_input_frames
        self.num_color_channels = num_color_channels
        self.temp1 = DenBlock(3, num_color_channels)
        self.temp2 = DenBlock(3, num_color_channels)
        self._engine = None
        self._twin = None
        self._twin_version = None

    def _state_version(self, own):
        return tuple(int(t._version) for t in own.values()) + tuple(t.data_ptr() for t in own.values())

    def _colour_twin(self):
        own = dict(self.state_dict())
        dev = next(self.parameters()).device
        if self._twin is None or next(self._twin[0].parameters()).device != dev:
            self._twin = (FastDVDnet(5, 3).to(dev),)          # in a tuple: NOT a sub-module (state_dict stays the gray model's)
            self._twin_version = None
        twin = self._twin[0]
        twin.train(self.training)
        version = self._state_version(own)
        if version != self._twin_version:
            with torch.no_grad():
                for k, dst in twin.state_dict().items():
                    src = own[k]
                    if src.shape == dst.shape:
                        dst.copy_(src)
                    elif k.endswith("inc.convblock.0.weight"):        # per frame group [y, sigma] -> [r, g, b, sigma]
                        dst.zero_()
                        dst[:, 0].copy_(src[:, 0])
                        dst[:, 3].copy_(src[:, 1])
                    elif k.endswith("outc.convblock.3.weight"):       # 32 -> 1 becomes the first of 32 -> 3
                        dst.zero_()
                        dst[0:1].copy_(src)
                    else:
                        raise RuntimeError("gray FastDVDnet: unexpected parameter shape for " + k)
            self._twin_version = version
        return twin

    def _restrict_twin(self):
        """Inverse of the embedding of ``_colour_twin``: the twin's (fine-tuned) weights back into the gray parameters, so
        that ``state_dict()`` holds them.  The twin's version is recorded after the write-back: it is not re-copied over
        itself on the next use."""
        own = dict(self.state_dict())
        with torch.no_grad():
            for k, src in self._twin[0].state_dict().items():
                dst = own[k]
                if src.shape == dst.shape:
                    dst.copy_(src)
                elif k.endswith("inc.convblock.0.weight"):            # [r, g, b, sigma] per frame group -> [y, sigma]
                    dst[:, 0].copy_(src[:, 0])
                    dst[:, 1].copy_(src[:, 3])
                elif k.endswith("outc.convblock.3.weight"):           # first of 32 -> 3 becomes 32 -> 1
                    dst.copy_(src[0:1])
                else:
                    raise RuntimeError("gray FastDVDnet: unexpected parameter shape for " + k)
        self._twin_version = self._state_version(own)

    def engine(self):
        from .engine import FastDVDnetEngine
        if self.num_color_channels == 1:
            return self._colour_twin().engine()
        if self._engine is None:
            self._engine = FastDVDnetEngine(self)
        return self._engine

    def forward(self, x, noise_map):
        """x [1,5*C,H,W] (5 frames stacked frame-major), noise_map [1,1,H,W] constant -> [1,C,H,W]."""
        if self.num_color_channels == 1:
            x3 = x.new_zeros((x.shape[0], 15, x.shape[2], x.shape[3]))
            x3[:, 0::3] = x
            return self.engine().forward_window(x3, noise_map)[:, 0:1]
        return self.engine().forward_window(x, noise_map)

    def __nchannel__(self):
        return self.num_color_channels
