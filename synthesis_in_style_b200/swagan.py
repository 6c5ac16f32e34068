"""SWAGAN generator with the reference's call surface (SURVEY.md §8(f) row 4), executed by the fused sm_100a plan.

Mirrors scf/networks/swagan/model.py:14-286: `HaarTransform`, `InverseHaarTransform`, the 12-channel wavelet `ToRGB` and
`Generator` (constructor signature, attributes, state-dict keys, random-init draw order, `forward` keywords and return
convention; the conv trunk stops at size / 2 and the image is the inverse Haar transform of the last skip).
`Generator.forward` is one `sis_generator_forward` call on a plan made by `sis_generator_create_swagan`: the conv trunk,
style MLP and labelling kernels of the StyleGAN2 plan (the trunk of SWAGAN-S is the trunk of StyleGAN2-S/2), and one
wavelet ToRGB launch per resolution, the last of which writes the image.  Everything else (activation capture, in-forward
labelling, `check`, `precision`, copies) is `model.Generator`'s.  Stand-alone, `ToRGB` is one `sis_wavelet_to_rgb` call
and the Haar modules are the drop-in `upfirdn2d` op.  Inference only; no CPU path.  GPU tests: tests/test_swagan.py,
tests/test_swagan_plan.py.
"""
import math

import torch
from torch import nn

from . import _lib
from .model import ConstantInput, ModulatedConv2d, StyledConv, _FirBuffer, _f32c, _Plan, _PlanGenerator, _StyleMLP, _stream
from .op import upfirdn2d


def get_haar_wavelet(in_channels=None):
    """swagan/model.py:14-25."""
    haar_wav_l = 1 / (2 ** 0.5) * torch.ones(1, 2)
    haar_wav_h = 1 / (2 ** 0.5) * torch.ones(1, 2)
    haar_wav_h[0, 0] = -1 * haar_wav_h[0, 0]
    return haar_wav_l.T * haar_wav_l, haar_wav_h.T * haar_wav_l, haar_wav_l.T * haar_wav_h, haar_wav_h.T * haar_wav_h


class HaarTransform(nn.Module):
    def __init__(self, in_channels):
        super().__init__()
        ll, lh, hl, hh = get_haar_wavelet(in_channels)
        self.register_buffer('ll', ll)
        self.register_buffer('lh', lh)
        self.register_buffer('hl', hl)
        self.register_buffer('hh', hh)

    def forward(self, input):
        return torch.cat([upfirdn2d(input, k, down=2) for k in (self.ll, self.lh, self.hl, self.hh)], 1)


class InverseHaarTransform(nn.Module):
    def __init__(self, in_channels):
        super().__init__()
        ll, lh, hl, hh = get_haar_wavelet(in_channels)
        self.register_buffer('ll', ll)
        self.register_buffer('lh', -lh)
        self.register_buffer('hl', -hl)
        self.register_buffer('hh', hh)

    def forward(self, input):
        ll, lh, hl, hh = input.chunk(4, 1)
        return (upfirdn2d(ll, self.ll, up=2, pad=(1, 0)) + upfirdn2d(lh, self.lh, up=2, pad=(1, 0))
                + upfirdn2d(hl, self.hl, up=2, pad=(1, 0)) + upfirdn2d(hh, self.hh, up=2, pad=(1, 0)))


class ToRGB(nn.Module):
    """swagan/model.py:71-98: 1x1 modulated conv (no demodulation) to 3 x 4 wavelet channels + bias; the skip is taken to
    the image domain, upsampled and transformed back."""

    def __init__(self, in_channel, style_dim, upsample=True, blur_kernel=(1, 3, 3, 1)):
        super().__init__()
        if upsample:
            self.iwt = InverseHaarTransform(3)
            p = len(blur_kernel) - 2
            self.upsample = _FirBuffer(blur_kernel, 4, up=2, pad=((p + 1) // 2 + 1, p // 2))
            self.dwt = HaarTransform(3)
        self.conv = ModulatedConv2d(in_channel, 3 * 4, 1, style_dim, demodulate=False)
        self.bias = nn.Parameter(torch.zeros(1, 3 * 4, 1, 1))

    def forward(self, input, style, skip=None):
        """swagan/model.py:84-98 through `sis_wavelet_to_rgb`: 1x1 modulated conv, bias and the skip chain in one pass."""
        x, st = _f32c(input, 'input'), _f32c(style, 'style')
        b, cin, h, _ = x.shape
        sk = _f32c(skip, 'skip') if skip is not None else None
        if sk is not None and (not hasattr(self, 'upsample') or tuple(sk.shape) != (b, 12, h // 2, h // 2)):
            raise RuntimeError('skip must be [B, 12, H/2, H/2] and the layer must have been built with upsample=True')
        taps = {}
        if hasattr(self, 'upsample'):
            for name in ('iwt', 'dwt'):
                m = getattr(self, name)
                taps[name] = _f32c(torch.stack([m.ll, m.lh, m.hl, m.hh]), f'{name} taps')
            taps['up'] = _f32c(self.upsample.kernel, 'upsample.kernel')
        mw, mb = _f32c(self.conv.modulation.weight.detach(), 'weight'), _f32c(self.conv.modulation.bias.detach(), 'bias')
        out = torch.empty(b, 12, h, h, device=x.device)
        with torch.cuda.device(x.device):
            _lib.check(_lib.load().sis_wavelet_to_rgb(
                _lib.ptr(x), b, cin, h, _lib.ptr(_f32c(self.conv.weight.detach(), 'weight')), _lib.ptr(mw), _lib.ptr(mb), mw.shape[1],
                _lib.ptr(st), _lib.ptr(_f32c(self.bias.detach(), 'bias')), _lib.ptr(sk), _lib.ptr(taps.get('iwt')),
                _lib.ptr(taps.get('up')), _lib.ptr(taps.get('dwt')), _lib.ptr(out), _stream(x)))
        return out


class Generator(_PlanGenerator):
    """swagan/model.py:101-286 on the plan of `sis_generator_create_swagan` (see `model.Generator` for the forward)."""

    _CREATE = 'sis_generator_create_swagan'

    def __init__(self, size, style_dim, n_mlp, channel_multiplier=2, blur_kernel=(1, 3, 3, 1), lr_mlp=0.01, precision='bf16x3'):
        super().__init__()
        self._require_plan_defaults(blur_kernel, lr_mlp)
        self.size, self.style_dim = size, style_dim
        self.n_mlp, self.channel_multiplier = n_mlp, channel_multiplier
        self.style = _StyleMLP(style_dim, n_mlp, lr_mlp)
        self.style._owner = (self,)   # tuple: not registered as a sub-module
        self.channels = self.get_channels(channel_multiplier)
        self.input = ConstantInput(self.channels[4])
        self.conv1 = StyledConv(self.channels[4], self.channels[4], 3, style_dim, blur_kernel=blur_kernel)
        self.to_rgb1 = ToRGB(self.channels[4], style_dim, upsample=False)
        self.log_size = int(math.log(size, 2)) - 1
        self.num_layers = (self.log_size - 2) * 2 + 1
        self.convs = nn.ModuleList()
        self.upsamples = nn.ModuleList()
        self.to_rgbs = nn.ModuleList()
        self.noises = nn.Module()
        in_channel = self.channels[4]
        for layer_idx in range(self.num_layers):
            res = (layer_idx + 5) // 2
            self.noises.register_buffer(f'noise_{layer_idx}', torch.randn(1, 1, 2 ** res, 2 ** res))
        for i in range(3, self.log_size + 1):
            out_channel = self.channels[2 ** i]
            self.convs.append(StyledConv(in_channel, out_channel, 3, style_dim, upsample=True, blur_kernel=blur_kernel))
            self.convs.append(StyledConv(out_channel, out_channel, 3, style_dim, blur_kernel=blur_kernel))
            self.to_rgbs.append(ToRGB(out_channel, style_dim))
            in_channel = out_channel
        self.iwt = InverseHaarTransform(3)
        self.n_latent = self.log_size * 2 - 2
        self.precision = precision
        for m in self.modules():
            if isinstance(m, ModulatedConv2d):
                m.precision = precision      # stand-alone layer calls follow the generator's precision
        self._plan = _Plan()
