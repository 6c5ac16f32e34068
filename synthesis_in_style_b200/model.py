"""StyleGAN2 generator with the reference's call surface, executed by the fused sm_100a plan in libsis_b200.

Mirrors the generator half of scf/networks/stylegan2/model.py (lines 15-561):
  * same constructor signature, attributes (`size, style_dim, channels, log_size, num_layers, n_latent, style,
    input, conv1, to_rgb1, convs, to_rgbs, noises`) and methods (`get_channels, make_noise, mean_latent,
    get_latent, forward`),
  * same parameter / buffer names, shapes and random-init draw order, so `g_ema` checkpoints load with
    `load_state_dict` and `torch.manual_seed(s); Generator(...)` reproduces the reference's weights,
  * `forward(...)` has the reference's keyword arguments and return convention
    (`(image, latent)`, `(image, {idx: activation})`, `(image, None)`).
The sub-modules are parameter containers: all arithmetic happens in `sis_generator_forward` (one C-ABI call per
batch, a fixed sequence of kernel launches on the current CUDA stream).  Inference only (the hot path runs under
`torch.no_grad()`, scf/utils/dataset_creation.py:49); there is no CPU path.
"""
import ctypes
import math
import random
import typing

import torch
from torch import nn

from . import _lib
from .op import FusedLeakyReLU

PRECISIONS = {'fp32': _lib.PRECISION_FP32, 'bf16x3': _lib.PRECISION_BF16X3}


class _Plan:
    """Owns the native `sis_generator*`.  Copies / pickles of a Generator start without a plan and rebuild it
    lazily from their own parameters."""

    def __init__(self):
        self.handle = None
        self.signature = None

    def __deepcopy__(self, memo):
        return _Plan()

    def __reduce__(self):
        return (_Plan, ())

    def __del__(self):
        try:
            if self.handle is not None:
                _lib.load().sis_generator_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


def make_kernel(k):
    """Normalised separable FIR taps (model.py:23-31)."""
    k = torch.tensor(k, dtype=torch.float32)
    if k.ndim == 1:
        k = k[None, :] * k[:, None]
    k /= k.sum()
    return k


def _stream(t):
    return _lib.current_stream_ptr(t.device)


def _f32c(t, name):
    _lib.require_cuda(t, name)
    return t.contiguous().float()


class PixelNorm(nn.Module):
    """model.py:15-20.  Inside `Generator.forward` it is part of the fused style-MLP launch; stand-alone it runs
    `sis_pixel_norm` (normalisation over dim 1 of a [N, D] input, the only way the generator uses it)."""

    def forward(self, input):
        x = _f32c(input, 'input')
        if x.dim() != 2:
            raise NotImplementedError('PixelNorm is implemented for [N, D] inputs (the style MLP)')
        out = torch.empty_like(x)
        with torch.cuda.device(x.device):
            _lib.check(_lib.load().sis_pixel_norm(_lib.ptr(x), _lib.ptr(out), x.shape[0], x.shape[1], _stream(x)))
        return out


class _FirBuffer(nn.Module):
    """Holds a `kernel` buffer under the reference's name (`blur.kernel`, `upsample.kernel`) and applies it like the
    reference's `Blur` (pad given) / `Upsample` (factor 2) modules when called (model.py:34-52, 76-92)."""

    def __init__(self, taps, gain, up=1, pad=(0, 0)):
        super().__init__()
        self.register_buffer('kernel', make_kernel(taps) * gain)
        self.up, self.pad = up, pad

    def forward(self, input):
        from .op import upfirdn2d
        return upfirdn2d(input, self.kernel, up=self.up, down=1, pad=self.pad)


class EqualLinear(nn.Module):
    """Parameters of model.py:133-150 (`weight = randn(out, in) / lr_mul`, `bias = bias_init`)."""

    def __init__(self, in_dim, out_dim, bias=True, bias_init=0, lr_mul=1, activation=None):
        super().__init__()
        self.weight = nn.Parameter(torch.randn(out_dim, in_dim).div_(lr_mul))
        self.bias = nn.Parameter(torch.zeros(out_dim).fill_(bias_init)) if bias else None
        self.activation = activation
        self.scale = (1 / math.sqrt(in_dim)) * lr_mul
        self.lr_mul = lr_mul

    def forward(self, input):
        """model.py:152-162 through `sis_equal_linear` (fused bias + leaky ReLU when `activation` is set)."""
        x = _f32c(input, 'input')
        x2 = x.reshape(-1, x.shape[-1])
        out = torch.empty(x2.shape[0], self.weight.shape[0], device=x.device)
        w = _f32c(self.weight.detach(), 'weight')
        b = _f32c(self.bias.detach(), 'bias') if self.bias is not None else None
        with torch.cuda.device(x.device):
            _lib.check(_lib.load().sis_equal_linear(_lib.ptr(x2), x2.shape[0], x2.shape[1], _lib.ptr(w), _lib.ptr(b), w.shape[0],
                                                    float(self.lr_mul), int(bool(self.activation)), _lib.ptr(out), _stream(x)))
        return out.reshape(*x.shape[:-1], w.shape[0])


class ModulatedConv2d(nn.Module):
    """Parameters of model.py:182-229."""

    def __init__(self, in_channel, out_channel, kernel_size, style_dim, demodulate=True, upsample=False,
                 blur_kernel=(1, 3, 3, 1)):
        super().__init__()
        self.eps = 1e-8
        self.kernel_size, self.in_channel, self.out_channel = kernel_size, in_channel, out_channel
        self.upsample, self.demodulate = upsample, demodulate
        if upsample:
            # Blur(kernel, pad=(pad0, pad1), upsample_factor=2), model.py:201-207: p = (4 - 2) - (3 - 1) = 0 -> pad (1, 1)
            p = (len(blur_kernel) - 2) - (kernel_size - 1)
            self.blur = _FirBuffer(blur_kernel, 4, up=1, pad=((p + 1) // 2 + 1, p // 2 + 1))
        self.scale = 1 / math.sqrt(in_channel * kernel_size ** 2)
        self.padding = kernel_size // 2
        self.weight = nn.Parameter(torch.randn(1, out_channel, in_channel, kernel_size, kernel_size))
        self.modulation = EqualLinear(style_dim, in_channel, bias_init=1)
        self.precision = 'bf16x3'

    def _run(self, input, style, noise=None, noise_weight=None, act_bias=None, activate=False):
        """One `sis_modulated_conv2d` call (model.py:237-278; with noise / bias / activation: StyledConv, :336-342)."""
        if self.kernel_size != 3:
            raise NotImplementedError('stand-alone ModulatedConv2d runs 3x3 kernels; the 1x1 case is ToRGB.forward')
        x, st = _f32c(input, 'input'), _f32c(style, 'style')
        b, cin, h, w_ = x.shape
        if h != w_ or cin != self.in_channel:
            raise RuntimeError(f'expected a square [B, {self.in_channel}, H, H] input')
        res_out = 2 * h if self.upsample else h
        out = torch.empty(b, self.out_channel, res_out, res_out, device=x.device)
        nz, nstride = None, 0
        if noise is not None:
            nz = _f32c(noise, 'noise')
            if nz.numel() == res_out * res_out:
                nstride = 0
            elif nz.numel() == b * res_out * res_out:
                nstride = res_out * res_out
            else:
                raise RuntimeError(f'noise must be [1,1,{res_out},{res_out}] or [{b},1,{res_out},{res_out}]')
        wt = _f32c(self.weight.detach(), 'weight')
        mw, mb = _f32c(self.modulation.weight.detach(), 'modulation.weight'), _f32c(self.modulation.bias.detach(), 'modulation.bias')
        blur = _f32c(self.blur.kernel, 'blur.kernel') if self.upsample else None
        nw = _f32c(noise_weight.detach(), 'noise.weight') if noise_weight is not None else None
        ab = _f32c(act_bias.detach(), 'activate.bias') if act_bias is not None else None
        with torch.cuda.device(x.device):
            _lib.check(_lib.load().sis_modulated_conv2d(
                _lib.ptr(x), b, cin, h, _lib.ptr(wt), self.out_channel, _lib.ptr(mw), _lib.ptr(mb), mw.shape[1], _lib.ptr(st),
                int(self.demodulate), int(self.upsample), _lib.ptr(blur), _lib.ptr(nz), nstride, _lib.ptr(nw), _lib.ptr(ab),
                int(activate), _lib.ptr(out), PRECISIONS[self.precision], _stream(x)))
        return out

    def forward(self, input, style):
        return self._run(input, style)


class NoiseInjection(nn.Module):
    def __init__(self):
        super().__init__()
        self.weight = nn.Parameter(torch.zeros(1))

    def forward(self, image, noise=None):
        """model.py:287-292: image + weight * noise (fresh per-sample noise when none is given)."""
        x = _f32c(image, 'image')
        b, c, h, w = x.shape
        if noise is None:
            noise = x.new_empty(b, 1, h, w).normal_()
        nz = _f32c(noise, 'noise')
        if nz.numel() not in (h * w, b * h * w):
            raise RuntimeError(f'noise must be [1,1,{h},{w}] or [{b},1,{h},{w}]')
        out = torch.empty_like(x)
        with torch.cuda.device(x.device):
            _lib.check(_lib.load().sis_noise_injection(_lib.ptr(x), _lib.ptr(nz), 0 if nz.numel() == h * w else h * w,
                                                       _lib.ptr(_f32c(self.weight.detach(), 'weight')), b, c, h, w, _lib.ptr(out), _stream(x)))
        return out


class ConstantInput(nn.Module):
    def __init__(self, channel, size=4):
        super().__init__()
        self.input = nn.Parameter(torch.randn(1, channel, size, size))

    def forward(self, input):
        """model.py:301-305: the learned constant repeated over the batch of `input`."""
        return self.input.repeat(input.shape[0], 1, 1, 1)


class StyledConv(nn.Module):
    """Parameters of model.py:308-334: conv, noise, activate."""

    def __init__(self, in_channel, out_channel, kernel_size, style_dim, upsample=False, blur_kernel=(1, 3, 3, 1),
                 demodulate=True):
        super().__init__()
        self.conv = ModulatedConv2d(in_channel, out_channel, kernel_size, style_dim, upsample=upsample,
                                    blur_kernel=blur_kernel, demodulate=demodulate)
        self.noise = NoiseInjection()
        self.activate = FusedLeakyReLU(out_channel)

    def forward(self, input, style, noise=None):
        """model.py:336-342: conv -> noise -> bias + leaky ReLU, one native call with the fused epilogue."""
        if noise is None:
            b, _, h, _ = input.shape
            r = 2 * h if self.conv.upsample else h
            noise = torch.empty(b, 1, r, r, device=input.device).normal_()
        return self.conv._run(input, style, noise=noise, noise_weight=self.noise.weight, act_bias=self.activate.bias, activate=True)


class ToRGB(nn.Module):
    """Parameters of model.py:345-353."""

    def __init__(self, in_channel, style_dim, upsample=True, blur_kernel=(1, 3, 3, 1)):
        super().__init__()
        if upsample:
            # Upsample(kernel, factor=2), model.py:34-52: kernel * factor**2, pad = ((p + 1) // 2 + 1, p // 2), p = 4 - 2
            p = len(blur_kernel) - 2
            self.upsample = _FirBuffer(blur_kernel, 4, up=2, pad=((p + 1) // 2 + 1, p // 2))
        self.conv = ModulatedConv2d(in_channel, 3, 1, style_dim, demodulate=False)
        self.bias = nn.Parameter(torch.zeros(1, 3, 1, 1))

    def forward(self, input, style, skip=None):
        """model.py:355-364 through `sis_to_rgb`: 1x1 modulated conv + bias + upsampled skip in one pass."""
        x, st = _f32c(input, 'input'), _f32c(style, 'style')
        b, cin, h, _ = x.shape
        out = torch.empty(b, 3, h, h, device=x.device)
        sk = _f32c(skip, 'skip') if skip is not None else None
        if sk is not None and (not hasattr(self, 'upsample') or tuple(sk.shape) != (b, 3, h // 2, h // 2)):
            raise RuntimeError('skip must be [B, 3, H/2, H/2] and the layer must have been built with upsample=True')
        upk = _f32c(self.upsample.kernel, 'upsample.kernel') if hasattr(self, 'upsample') else None
        mw, mb = _f32c(self.conv.modulation.weight.detach(), 'weight'), _f32c(self.conv.modulation.bias.detach(), 'bias')
        with torch.cuda.device(x.device):
            _lib.check(_lib.load().sis_to_rgb(_lib.ptr(x), b, cin, h, _lib.ptr(_f32c(self.conv.weight.detach(), 'weight')), _lib.ptr(mw),
                                              _lib.ptr(mb), mw.shape[1], _lib.ptr(st), _lib.ptr(_f32c(self.bias.detach(), 'bias')),
                                              _lib.ptr(sk), _lib.ptr(upk), _lib.ptr(out), _stream(x)))
        return out


class _StyleMLP(nn.Module):
    """`Generator.style` (model.py:383-392): PixelNorm at index 0, EqualLinear at 1..n_mlp (keys `style.{i}.*`).
    Calling it runs the fused style-MLP of the owning generator."""

    def __init__(self, style_dim, n_mlp, lr_mlp):
        super().__init__()
        self.add_module('0', PixelNorm())
        for i in range(n_mlp):
            self.add_module(str(i + 1), EqualLinear(style_dim, style_dim, lr_mul=lr_mlp, activation='fused_lrelu'))
        self._owner = None

    def forward(self, z):
        return self._owner[0]._style(z)


class _PlanGenerator(nn.Module):
    """The native plan behind a generator with the reference's call surface: the StyleGAN2 `Generator` below and
    `swagan.Generator`.  A subclass builds the reference's module tree (the state dict the plan reads) with the attributes
    `size, style_dim, n_mlp, channel_multiplier, channels, log_size, num_layers, n_latent, precision, input`, a `_StyleMLP`
    as `style` and `_plan = _Plan()`, and names the C-ABI call that creates its plan in `_CREATE`."""

    _CREATE = 'sis_generator_create'

    @staticmethod
    def _require_plan_defaults(blur_kernel, lr_mlp):
        if list(blur_kernel) != [1, 3, 3, 1]:
            raise NotImplementedError('the fused plan is built for the reference default blur_kernel=[1, 3, 3, 1]')
        if lr_mlp != 0.01:
            raise NotImplementedError('the fused plan is built for the reference default lr_mlp=0.01')

    # ------------------------------------------------------------------ reference helpers
    @staticmethod
    def get_channels(channel_multiplier=2) -> typing.Dict[int, int]:
        return {4: 512, 8: 512, 16: 512, 32: 512, 64: 256 * channel_multiplier, 128: 128 * channel_multiplier,
                256: 64 * channel_multiplier, 512: 32 * channel_multiplier, 1024: 16 * channel_multiplier}

    def make_noise(self) -> typing.List[torch.Tensor]:
        """model.py:457-466: one 4x4 map, then two per resolution, [1,1,H,W] on the generator's device."""
        device = self.input.input.device
        noises = [torch.randn(1, 1, 4, 4, device=device)]
        for i in range(3, self.log_size + 1):
            for _ in range(2):
                noises.append(torch.randn(1, 1, 2 ** i, 2 ** i, device=device))
        return noises

    def mean_latent(self, n_latent):
        """model.py:468-474."""
        latent_in = torch.randn(n_latent, self.style_dim, device=self.input.input.device)
        return self.style(latent_in).mean(0, keepdim=True)

    def get_latent(self, input):
        return self.style(input)

    def activation_shape(self, idx: int):
        """(channels, resolution) of captured activation `idx` (0 .. n_latent-1)."""
        res = 4 if idx <= 1 else 2 ** ((idx - 2) // 2 + 3)
        return self.channels[res], res

    # ------------------------------------------------------------------ native plan management
    @property
    def _handle(self):
        return self._plan.handle

    def _named_state(self):
        for name, t in self.named_parameters():
            yield name, t
        for name, t in self.named_buffers():
            yield name, t

    def _sync(self):
        """(Re)bind the state dict to the native plan when a tensor was replaced or modified in place."""
        lib = _lib.load()
        state = list(self._named_state())
        dev = self.input.input.device
        for name, t in state:
            if not t.is_cuda:
                raise RuntimeError(f'{name} must be a CUDA tensor (libsis_b200 has no CPU path)')
            if t.device != dev:
                raise RuntimeError('all generator parameters must live on one CUDA device')
            if t.dtype != torch.float32:
                raise RuntimeError(f'{name}: the fused plan takes fp32 parameters (got {t.dtype})')
        signature = tuple((name, t.data_ptr(), t._version, tuple(t.shape)) for name, t in state)
        if self._plan.handle is not None and signature == self._plan.signature:
            return dev
        with torch.cuda.device(dev):
            if self._plan.handle is None:
                h = ctypes.c_void_p()
                _lib.check(getattr(lib, self._CREATE)(self.size, self.style_dim, self.n_mlp, self.channel_multiplier,
                                                      ctypes.byref(h)))
                self._plan.handle = h
            keep = []
            for name, t in state:
                tc = t.detach().contiguous()
                keep.append(tc)
                _lib.check(lib.sis_generator_set_param(self._handle, name.encode(), _lib.ptr(tc), tc.numel()))
            _lib.check(lib.sis_generator_prepare(self._handle, _lib.current_stream_ptr(dev)))
        self._plan.signature = signature
        return dev

    def check(self):
        """Drain the current stream and raise if a bounded device-side wait of the tcgen05 kernels gave up
        (`sis_generator_check`); tests and bench.py call it after a run."""
        if self._plan.handle is None:
            return
        dev = self.input.input.device
        with torch.cuda.device(dev):
            _lib.check(_lib.load().sis_generator_check(self._handle, _lib.current_stream_ptr(dev)))

    def _style(self, z: torch.Tensor) -> torch.Tensor:
        _lib.require_cuda(z, 'input')
        dev = self._sync()
        z2 = z.reshape(-1, self.style_dim).contiguous().float()
        w = torch.empty_like(z2)
        with torch.cuda.device(dev):
            _lib.check(_lib.load().sis_generator_style(self._handle, _lib.ptr(z2), _lib.ptr(w), z2.shape[0],
                                                       _lib.current_stream_ptr(dev)))
        return w.reshape(z.shape)

    # ------------------------------------------------------------------ forward
    def forward(self, styles, return_latents=False, inject_index=None, truncation=1, truncation_latent=None,
                input_is_latent=False, noise=None, randomize_noise=True, return_intermediate_activations=False,
                capture_layers=None, label_jobs=None):
        """Same arguments / returns as the reference (model.py:479-561).  Two optional extensions (not in the reference):
        `capture_layers` restricts which activation indices are materialised when `return_intermediate_activations`;
        `label_jobs` (a list of `labelling.LabelJobSpec`) labels activations inside the same native call, fused with
        the StyleGAN2 ToRGB pass where both read the same tensor."""
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            # The fused plan is inference-only.  Running silently without a graph would be a wrong gradient.
            raise RuntimeError('Generator.forward of synthesis_in_style_b200 is inference-only: call it under '
                               'torch.no_grad() (the reference hot path does, utils/dataset_creation.py:49)')
        dev = self._sync()
        lib = _lib.load()
        styles = list(styles)
        if len(styles) not in (1, 2):
            raise RuntimeError('styles must hold one or two tensors')
        for s in styles:
            _lib.require_cuda(s, 'styles')
        wplus = len(styles) == 1 and styles[0].ndim == 3 and input_is_latent
        if styles[0].ndim == 3 and not wplus:
            raise RuntimeError('a [B, n_latent, style_dim] style needs input_is_latent=True and no second style')
        batch = styles[0].shape[0]
        st = [s.contiguous().float() for s in styles]
        if wplus and tuple(st[0].shape[1:]) != (self.n_latent, self.style_dim):
            raise RuntimeError(f'W+ latent must be [B, {self.n_latent}, {self.style_dim}]')

        # noise (model.py:494-500 and NoiseInjection.forward :287-292)
        if noise is None:
            if randomize_noise:
                noise = []
                for layer in range(self.num_layers):
                    res = 2 ** ((layer + 5) // 2)
                    noise.append(torch.empty(batch, 1, res, res, device=dev).normal_())
            else:
                noise = [getattr(self.noises, f'noise_{i}') for i in range(self.num_layers)]
        noise = list(noise)
        if len(noise) != self.num_layers:
            raise RuntimeError(f'noise must hold {self.num_layers} maps')
        noise_t, strides = [], []
        for layer, n in enumerate(noise):
            res = 2 ** ((layer + 5) // 2)
            if n is None:
                n = torch.empty(batch, 1, res, res, device=dev).normal_()
            _lib.require_cuda(n, 'noise')
            if n.numel() == res * res:
                strides.append(0)
            elif n.numel() == batch * res * res:
                strides.append(res * res)
            else:
                raise RuntimeError(f'noise[{layer}] must be [1,1,{res},{res}] or [{batch},1,{res},{res}]')
            noise_t.append(n.contiguous().float())

        if len(styles) == 2 and inject_index is None:
            inject_index = random.randint(1, self.n_latent - 1)     # model.py:522-523
        tl = None
        if truncation < 1:
            if truncation_latent is None:
                raise RuntimeError('truncation < 1 needs truncation_latent')
            _lib.require_cuda(truncation_latent, 'truncation_latent')
            tl = truncation_latent.reshape(-1, self.style_dim).contiguous().float()
            if tl.shape[0] not in (1, batch):
                raise RuntimeError('truncation_latent must be [1, style_dim] or [B, style_dim]')

        image = torch.empty(batch, 3, self.size, self.size, device=dev)
        latent_out = torch.empty(batch, self.n_latent, self.style_dim, device=dev) if return_latents else None
        acts = None
        if return_intermediate_activations and not return_latents:
            wanted = range(self.n_latent) if capture_layers is None else sorted(set(int(i) for i in capture_layers))
            acts = {}
            for idx in wanted:
                c, res = self.activation_shape(idx)
                acts[idx] = torch.empty(batch, c, res, res, device=dev)

        args = _lib.ForwardArgs()
        args.batch = batch
        args.n_styles = len(st)
        args.d_styles[0] = st[0].data_ptr()
        args.d_styles[1] = st[1].data_ptr() if len(st) == 2 else None
        args.input_is_latent = int(bool(input_is_latent))
        args.styles_are_wplus = int(wplus)
        args.inject_index = int(inject_index) if inject_index is not None else self.n_latent
        args.truncation = float(truncation)
        args.d_truncation_latent = tl.data_ptr() if tl is not None else None
        args.truncation_latent_rows = tl.shape[0] if tl is not None else 0
        noise_ptrs = (ctypes.c_void_p * self.num_layers)(*[n.data_ptr() for n in noise_t])
        noise_strides = (ctypes.c_int64 * self.num_layers)(*strides)
        args.d_noise = ctypes.cast(noise_ptrs, ctypes.POINTER(ctypes.c_void_p))
        args.noise_batch_stride = ctypes.cast(noise_strides, ctypes.POINTER(ctypes.c_int64))
        args.d_image = image.data_ptr()
        args.d_latent_out = latent_out.data_ptr() if latent_out is not None else None
        act_ptrs = None
        if acts is not None:
            act_ptrs = (ctypes.c_void_p * self.n_latent)(*[acts[i].data_ptr() if i in acts else None
                                                           for i in range(self.n_latent)])
            args.d_activations = ctypes.cast(act_ptrs, ctypes.POINTER(ctypes.c_void_p))
        else:
            args.d_activations = None
        c_jobs = None
        if label_jobs:
            c_jobs = (_lib.LabelJob * len(label_jobs))()
            for cj, spec in zip(c_jobs, label_jobs):
                spec.fill(cj)
            args.n_label_jobs = len(label_jobs)
            args.label_jobs = ctypes.cast(c_jobs, ctypes.POINTER(_lib.LabelJob))
        else:
            args.n_label_jobs = 0
            args.label_jobs = None
        if self.precision not in PRECISIONS:
            raise RuntimeError(f'unknown precision {self.precision!r} (use one of {sorted(PRECISIONS)})')
        args.precision = PRECISIONS[self.precision]
        if batch > 0:
            with torch.cuda.device(dev):
                _lib.check(lib.sis_generator_forward(self._handle, ctypes.byref(args), _lib.current_stream_ptr(dev)))
        if return_latents:
            return image, latent_out
        if return_intermediate_activations:
            return image, acts
        return image, None


class Generator(_PlanGenerator):
    def __init__(self, size, style_dim, n_mlp, channel_multiplier=2, blur_kernel=(1, 3, 3, 1), lr_mlp=0.01,
                 precision='bf16x3'):
        super().__init__()
        self._require_plan_defaults(blur_kernel, lr_mlp)
        self.size, self.style_dim = size, style_dim
        self.n_mlp, self.channel_multiplier = n_mlp, channel_multiplier
        self.precision = precision
        self.style = _StyleMLP(style_dim, n_mlp, lr_mlp)
        self.style._owner = (self,)   # tuple: not registered as a sub-module
        self.channels = self.get_channels(channel_multiplier)
        self.input = ConstantInput(self.channels[4])
        self.conv1 = StyledConv(self.channels[4], self.channels[4], 3, style_dim, blur_kernel=blur_kernel)
        self.to_rgb1 = ToRGB(self.channels[4], style_dim, upsample=False)
        self.log_size = int(math.log(size, 2))
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
        self.n_latent = self.log_size * 2 - 2
        for m in self.modules():
            if isinstance(m, ModulatedConv2d):
                m.precision = precision      # stand-alone layer calls follow the generator's precision
        self._plan = _Plan()
