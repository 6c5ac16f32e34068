"""Every conv-family kernel instantiation of the native library, checked against a float64 restatement of the layer.

`tc_modconv` picks one of several dozen kernel instantiations from the layer's shape and the batch size (halo rule,
N tile, cost model, CTA pairs), and `sis_modulated_conv2d` falls back to the fp32 CUDA-core kernel for channel counts
that are not multiples of 32.  Each row of `ROWS` is a (B, Cin, Cout, H, upsample) call through `ModulatedConv2d` /
`StyledConv`, with the exact set of conv-family kernels that call launches.  The set is asserted from the profiler's
kernel names, so a change of the dispatch rules that moves a row to another kernel fails here, and
`test_every_compiled_conv_kernel_has_a_row` makes the table cover every instantiation compiled into the library.

The bound is per element, normalised by the root-sum-square of the products that feed the element:
    |got - ref| <= tau * rss,   rss = d * sqrt(sum over taps and channels of (x s)^2 (scale W)^2 (blur tap)^2).
bf16x3 (x s and scale W split into bf16 hi + lo, hi hi + hi lo + lo hi summed in fp32) sits near 2e-5 on this metric
and the fp32 CUDA-core conv near 1e-6; `test_bound_separates_bf16x3_from_planted_faults` (CPU) shows that tau keeps
the clean emulation in and typical kernel faults (a dropped K chunk's lo terms, a missing cross term, one channel off by
2^-10, a dropped tap, a pixel from the neighbouring sample) out.
"""
import math
import os
import re
import subprocess
import time
from collections import namedtuple

import pytest
import torch
import torch.nn.functional as F

from oracle import stylegan2_oracle as so
from synthesis_in_style_b200 import _lib
from synthesis_in_style_b200 import model as M

TAU = {'bf16x3': 2e-4, 'fp32': 2e-5}
STYLE_DIM = 64
FAMILY = re.compile(r'^(modconv_tc|blur_act_split|modconv3x3_simt|blur_noise_act)')


# ------------------------------------------------------------------------------------------------- the case table

def tc(bn, bk, cg):
    return f'modconv_tc_kernel<{bn}, {bk}, {cg}>'


def halo(bn, cg, bk, up4):
    return f'modconv_tc_halo_kernel<{bn}, {cg}, {bk}, {"true" if up4 else "false"}>'


def rw(bn, bk, up4):
    return f'modconv_tc_halo_rw_kernel<{bn}, {bk}, {"true" if up4 else "false"}>'


def blur(sep, cb):
    return f'blur_act_split_kernel<{"true" if sep else "false"}, {cb}>'


HALO_T = 'modconv_tc_halo_t_kernel'
SIMT = 'modconv3x3_simt_kernel'
BLUR_SIMT = 'blur_noise_act_kernel'

Row = namedtuple('Row', 'id B cin cout H up kernels demod nonsep precision')


def row(id_, B, cin, cout, H, up, kernels, demod=True, nonsep=False, precision='bf16x3'):
    return Row(id_, B, cin, cout, H, up, frozenset(kernels), demod, nonsep, precision)


# "tiles" below are the pixel tiles (M = 128) the CTA-pair launch splits into pairs; an odd count leaves the last pair
# with an idle second CTA.  Plain halo layers always have an even count (H/16 x H/8 = 2 (H/16)^2 tiles per sample).
ROWS = [
    # per-tap kernel, single CTAs: the 4^2 / 8^2 / 12^2 plain layers (N tile from the cost model); at 4^2 and 12^2 one
    # 128-pixel run spans several samples
    row('tc<32,64,1>', 3, 512, 512, 4, False, {tc(32, 64, 1)}),
    row('tc<32,32,1>', 2, 32, 32, 4, False, {tc(32, 32, 1)}),
    row('tc<64,64,1>', 49, 64, 192, 8, False, {tc(64, 64, 1)}, demod=False),
    row('tc<64,32,1>', 49, 32, 192, 8, False, {tc(64, 32, 1)}),
    row('tc<128,64,1>', 37, 64, 512, 8, False, {tc(128, 64, 1)}),
    row('tc<128,32,1>', 37, 32, 512, 8, False, {tc(128, 32, 1)}),
    row('tc<256,64,1>', 33, 64, 512, 12, False, {tc(256, 64, 1)}),
    row('tc<256,32,1>', 33, 32, 512, 12, False, {tc(256, 32, 1)}),
    # per-tap kernel, CTA pairs: 4-phase up-convs, each phase padded to the largest phase's pair tiles
    row('tc<64,64,2>-up', 44, 64, 192, 8, True, {tc(64, 64, 2), blur(True, 64)}),            # phase tiles 28/25/25/22
    row('tc<64,32,2>-up', 44, 32, 192, 8, True, {tc(64, 32, 2), blur(True, 64)}),            # phase tiles 28/25/25/22
    row('tc<128,64,2>-up', 61, 64, 128, 12, True, {tc(128, 64, 2), blur(True, 64)}),         # phase tiles 81/75/75/69
    row('tc<128,32,2>-up', 61, 32, 128, 12, True, {tc(128, 32, 2), blur(True, 64)}),         # phase tiles 81/75/75/69
    row('tc<256,64,2>-up', 61, 64, 256, 12, True, {tc(256, 64, 2), blur(True, 64)}),         # phase tiles 81/75/75/69
    row('tc<256,32,2>-up', 61, 32, 256, 12, True, {tc(256, 32, 2), blur(True, 64)}, demod=False),
    row('tc<128,32,2>-plain', 264, 32, 128, 12, False, {tc(128, 32, 2)}),                     # 297 tiles
    # halo kernel, plain 3x3 (H % 16 == 0)
    row('halo<32,1,64,F>', 1, 64, 32, 16, False, {halo(32, 1, 64, False)}),
    row('halo<32,1,32,F>', 1, 32, 64, 16, False, {halo(32, 1, 32, False)}),
    row('halo<64,1,32,F>', 19, 32, 64, 32, False, {halo(64, 1, 32, False)}),
    row('halo<64,2,32,F>', 37, 32, 64, 32, False, {halo(64, 2, 32, False)}),                 # 296 tiles
    row('halo<64,1,64,F>', 37, 64, 128, 16, False, {halo(64, 1, 64, False)}, demod=False),
    row('halo<64,2,64,F>', 37, 64, 64, 32, False, {halo(64, 2, 64, False)}),                 # 296 tiles
    row('halo<128,1,64,F>', 37, 64, 256, 16, False, {halo(128, 1, 64, False)}),
    row('halo<128,2,64,F>', 17, 64, 128, 48, False, {halo(128, 2, 64, False)}),              # 306 tiles
    row('halo<256,1,64,F>', 37, 64, 512, 16, False, {halo(256, 1, 64, False)}),
    row('halo<256,2,64,F>', 37, 64, 256, 32, False, {halo(256, 2, 64, False)}),              # 296 tiles
    # resident-weight halo kernels
    row('rw<32,32,F>', 1, 32, 32, 16, False, {rw(32, 32, False)}, demod=False),
    row('rw<32,64,T>-up', 1, 64, 32, 8, True, {rw(32, 64, True), blur(True, 64)}),
    # 4-phase halo kernel of the Cout <= 64 up-convs; its tiles cover the (H+1)^2 grid
    row('halo<32,1,32,T>-up', 1, 32, 32, 8, True, {halo(32, 1, 32, True), blur(True, 64)}),
    row('halo<32,1,64,T>-up', 1, 128, 32, 8, True, {halo(32, 1, 64, True), blur(True, 64)}),
    row('halo<64,1,32,T>-up', 1, 32, 64, 8, True, {halo(64, 1, 32, True), blur(True, 64)}),
    row('halo<64,1,64,T>-up', 1, 64, 64, 8, True, {halo(64, 1, 64, True), blur(True, 64)}, demod=False),
    row('halo<64,2,32,T>-up', 21, 32, 64, 32, True, {halo(64, 2, 32, True), blur(True, 64)}),   # 315 tiles
    row('halo<64,2,64,T>-up', 50, 64, 64, 16, True, {halo(64, 2, 64, True), blur(True, 64)}),   # 300 tiles
    # the blur pass: 32-channel blocks for Cout % 64 != 0 with a >= 32-wide output; the generic 16-tap path for a
    # non-separable `blur.kernel` (an asymmetric one, so that the tap flip is checked too)
    row('blur<T,32>-up', 2, 32, 32, 16, True, {halo(32, 1, 32, True), blur(True, 32)}),
    row('blur<F,64>-up', 1, 64, 64, 8, True, {halo(64, 1, 64, True), blur(False, 64)}, nonsep=True),
    row('blur<F,32>-up', 1, 32, 32, 16, True, {halo(32, 1, 32, True), blur(False, 32)}, nonsep=True),
    # transposed-product halo kernel: Cout = 128 with H % 32 == 0; up-convs add the per-tap border strips
    row('halo_t', 1, 32, 128, 32, False, {HALO_T}, demod=False),
    row('halo_t-96', 3, 64, 128, 96, False, {HALO_T}),
    row('halo_t+strips-up', 2, 64, 128, 32, True, {HALO_T, tc(128, 64, 1), blur(True, 64)}),
    row('halo_t+strips-up-128', 1, 64, 128, 128, True, {HALO_T, tc(128, 64, 1), blur(True, 64)}),
    # fp32 CUDA-core conv: under fp32, and under bf16x3 when a channel count is not a multiple of 32
    row('simt-fp32', 2, 48, 40, 12, False, {SIMT}, demod=False, precision='fp32'),
    row('simt-bf16x3', 2, 48, 40, 12, False, {SIMT}),
    row('simt-fp32-up', 2, 48, 40, 12, True, {SIMT, BLUR_SIMT}, precision='fp32'),
    row('simt-bf16x3-up', 2, 48, 40, 12, True, {SIMT, BLUR_SIMT}, nonsep=True),
]


# ------------------------------------------------------------------------------------------ float64 restatement

def nonseparable_blur():
    """A 4x4 blur that is neither separable nor symmetric (sum 4, like the reference's upsampling blur)."""
    k = so.make_kernel([1, 3, 3, 1]) * 4
    k = k + torch.tensor([[0.05, -0.02, 0.0, 0.01], [0.0, 0.03, -0.04, 0.0], [0.02, 0.0, 0.0, -0.03], [-0.01, 0.0, 0.04, 0.0]])
    return k


def restate(x, style, weight, mod_w, mod_b, demodulate, blur_k=None):
    """ModulatedConv2d.forward in float64 on the inputs' device, and the root-sum-square of the products behind each
    output element.  The modulated conv is conv(x * s, scale * W) * d; with `blur_k` it is the stride-2 transposed conv
    followed by the 4x4 blur (true convolution, pad (1, 1)), the reference's upsampling layer."""
    x, style, weight, mod_w, mod_b = (t.double() for t in (x, style, weight, mod_w, mod_b))
    w = weight.reshape(weight.shape[-4:]) * (1.0 / math.sqrt(weight.shape[-3] * 9))       # [Cout, Cin, 3, 3]
    s = style @ (mod_w * (1.0 / math.sqrt(mod_w.shape[1]))).t() + mod_b                   # EqualLinear, lr_mul 1
    if demodulate:
        d = torch.rsqrt((s * s) @ (w * w).sum((2, 3)).t() + 1e-8)                          # [B, Cout]
    else:
        d = torch.ones(x.shape[0], w.shape[0], dtype=torch.float64, device=x.device)
    xs = x * s[:, :, None, None]
    if blur_k is None:
        out, sq = F.conv2d(xs, w, padding=1), F.conv2d(xs * xs, w * w, padding=1)
    else:
        out = F.conv_transpose2d(xs, w.transpose(0, 1), stride=2)
        sq = F.conv_transpose2d(xs * xs, (w * w).transpose(0, 1), stride=2)
        k = torch.flip(blur_k.double(), [0, 1])
        c = out.shape[1]
        out = F.conv2d(F.pad(out, (1, 1, 1, 1)), k.expand(c, 1, 4, 4), groups=c)
        sq = F.conv2d(F.pad(sq, (1, 1, 1, 1)), (k * k).expand(c, 1, 4, 4), groups=c)
    return out * d[:, :, None, None], sq.sqrt() * d[:, :, None, None]


def restate_styled(ref, noise, noise_w, bias):
    """StyledConv after the conv: + noise_w * noise, + bias, leaky ReLU(0.2) * sqrt(2), in float64; and the size of
    the pre-activation terms (for the fp32 rounding of the epilogue)."""
    pre = ref + float(noise_w) * noise.double() + bias.double()[None, :, None, None]
    mag = ref.abs() + abs(float(noise_w)) * noise.double().abs() + bias.double().abs()[None, :, None, None]
    return torch.where(pre > 0, pre, 0.2 * pre) * math.sqrt(2.0), mag


def normalised_error(got, ref, rss):
    return float(((got.double() - ref).abs() / rss.clamp_min(1e-300)).max())


def conv_params(module):
    c = module.conv if isinstance(module, M.StyledConv) else module
    return (c.weight.detach(), c.modulation.weight.detach(), c.modulation.bias.detach(), c.demodulate,
            c.blur.kernel if c.upsample else None)


# ------------------------------------------------------------------------------------------------ CPU self-checks

def split_bf16(t):
    hi = t.bfloat16().float()
    return hi, (t - hi).bfloat16().float()


def emulate_bf16x3(x, style, weight, mod_w, mod_b, fault=None):
    """The tcgen05 conv's arithmetic on the CPU: x s and scale W split into bf16 hi + lo, hi hi + hi lo + lo hi in fp32,
    times d, for a plain 3x3 layer; `fault` plants one of the errors the bound must catch."""
    cin = weight.shape[2]
    s = (style @ (mod_w / math.sqrt(mod_w.shape[1])).t() + mod_b).float()
    w = weight[0].float() / math.sqrt(cin * 9)
    d = torch.rsqrt((s * s) @ (w * w).sum((2, 3)).t() + 1e-8)
    xh, xl = split_bf16(x.float() * s[:, :, None, None])
    wh, wl = split_bf16(w)
    if fault == 'chunk_lo':                       # lo terms of K chunk 1 (input channels 64..127) dropped
        xl, wl = xl.clone(), wl.clone()
        xl[:, 64:128] = 0
        wl[:, 64:128] = 0
    out = F.conv2d(xh, wh, padding=1) + F.conv2d(xh, wl, padding=1)
    if fault != 'x_lo_w_hi':
        out = out + F.conv2d(xl, wh, padding=1)
    if fault == 'tap_last_column':                # tap (ky, kx) = (1, 0) missing in the last output column
        tap = torch.zeros_like(wh)
        tap[:, :, 1, 0] = 1
        out[..., -1] -= F.conv2d(xh, wh * tap, padding=1)[..., -1]
    out = out * d[:, :, None, None]
    if fault == 'channel_ulp':
        out[:, 5] *= 1 + 2 ** -10
    if fault == 'neighbour_pixel':
        out[1, :, 3, 4] = out[2, :, 3, 4]
    return out


def make_layer(cin, cout, up, seed, nonsep=False, demod=True):
    torch.manual_seed(seed)
    m = M.StyledConv(cin, cout, 3, STYLE_DIM, upsample=up, demodulate=demod)
    with torch.no_grad():
        m.noise.weight.fill_(0.37)
        m.activate.bias.normal_(0, 0.1)
        if nonsep:
            m.conv.blur.kernel.copy_(nonseparable_blur())
    return m


def test_bound_separates_bf16x3_from_planted_faults():
    torch.manual_seed(0)
    B, cin, cout, H = 3, 512, 64, 8
    m = make_layer(cin, cout, False, seed=5)
    x, style = torch.randn(B, cin, H, H), torch.randn(B, STYLE_DIM)
    w, mw, mb, _, _ = conv_params(m)
    ref, rss = restate(x, style, w, mw, mb, True)
    clean = normalised_error(emulate_bf16x3(x, style, w, mw, mb), ref, rss)
    assert clean <= TAU['bf16x3'] / 5, clean
    scores = {f: normalised_error(emulate_bf16x3(x, style, w, mw, mb, fault=f), ref, rss)
              for f in ('chunk_lo', 'x_lo_w_hi', 'channel_ulp', 'tap_last_column', 'neighbour_pixel')}
    print(f'bf16x3 emulation {clean:.2e}; planted faults ' + ', '.join(f'{k} {v:.2e}' for k, v in scores.items()))
    for fault, score in scores.items():
        assert score > TAU['bf16x3'], (fault, score)
    # the fp32 conv sits an order of magnitude below the fp32 bound
    s = style @ (mw / math.sqrt(STYLE_DIM)).t() + mb
    wf = w[0] / math.sqrt(cin * 9)
    d = torch.rsqrt((s * s) @ (wf * wf).sum((2, 3)).t() + 1e-8)
    fp32 = F.conv2d(x * s[:, :, None, None], wf, padding=1) * d[:, :, None, None]
    assert normalised_error(fp32, ref, rss) <= TAU['fp32'] / 5


@pytest.mark.parametrize('up,demod,nonsep', [(False, True, False), (False, False, False), (True, True, False),
                                             (True, False, True), (True, True, True)])
def test_restatement_matches_the_oracle(up, demod, nonsep):
    """The float64 restatement is the reference's ModulatedConv2d / StyledConv (flip, padding, blur placement)."""
    m = make_layer(24, 16, up, seed=11, nonsep=nonsep, demod=demod)
    sd = {f'L.{k}': v for k, v in m.state_dict().items()}
    torch.manual_seed(1)
    B, H = 3, 7
    x, style = torch.randn(B, 24, H, H), torch.randn(B, STYLE_DIM)
    r = 2 * H if up else H
    noise = torch.randn(B, 1, r, r)
    ref, rss = restate(x, style, *conv_params(m))
    want = so.modulated_conv2d(sd, 'L.conv', x, style, demodulate=demod, upsample=up)
    assert ref.shape == want.shape and normalised_error(want, ref, rss) <= 1e-5
    if nonsep:   # the asymmetric blur tells the flipped taps from the unflipped ones
        w, mw, mb, dm, k = conv_params(m)
        unflipped, _ = restate(x, style, w, mw, mb, dm, torch.flip(k, [0, 1]))
        assert normalised_error(unflipped, ref, rss) > 1e-2
    if demod:
        sty, mag = restate_styled(ref, noise, sd['L.noise.weight'], sd['L.activate.bias'])
        want_sty = so.styled_conv(sd, 'L', x, style, noise, upsample=up)
        assert float((want_sty.double() - sty).abs().max()) <= 1e-5 * float(mag.max())


def test_every_compiled_conv_kernel_has_a_row():
    """The conv-family kernels compiled into the library (their host stubs, listed by `nm -C`) are exactly the ones the
    table launches: a new variant needs a row, and a variant no row reaches should not be shipped."""
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip('the native library has not been built')
    res = subprocess.run(['nm', '-C', _lib.LIB_PATH], capture_output=True, text=True)
    assert res.returncode == 0 and res.stdout, f'cannot list the symbols of {_lib.LIB_PATH}: {res.stderr.strip()}'
    compiled = set()
    for line in res.stdout.splitlines():
        parts = line.split(' ', 2)
        if len(parts) == 3 and parts[1] in 'tTwW':
            m = re.match(r'(?:void )?sis::(\w+(?:<[^()]*>)?)\(', parts[2])
            if m and FAMILY.match(m.group(1)) and m.group(1).split('<')[0].endswith('_kernel'):
                compiled.add(m.group(1))
    covered = set().union(*(r.kernels for r in ROWS))
    assert compiled, 'no conv-family kernel symbols found'
    assert compiled - covered == set(), f'compiled but launched by no row: {sorted(compiled - covered)}'
    assert covered - compiled == set(), f'in the table but not compiled: {sorted(covered - compiled)}'


# ---------------------------------------------------------------------------------------------------- GPU rows

def launched_conv_kernels(fn):
    """Run `fn` once under the profiler; the `name<args>` of every conv-family kernel it launched."""
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = set()
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        m = re.search(r'sis::(\w+(?:<[^()]*>)?)\(', e.name)
        if m and FAMILY.match(m.group(1)):
            names.add(m.group(1))
    return out, names


def poison_shapes(r):
    """Calls at the row's batch that fit the operand planes the row sized (B x Cin x res^2 bf16 elements, res the
    power of two >= H) without growing them, but lay the planes out differently: another Cin and H covering as much of
    them as possible (the row's own shape where none fits).  Up rows also refill the up-conv scratch at the row's own
    shape.  The poison stays on the same side of the tcgen05 / CUDA-core split as the row."""
    res = 4
    while res < r.H:
        res *= 2
    cands = [(c * h * h, c, h) for c in (r.cin // 2, 2 * r.cin, 3 * r.cin) if (c % 32 == 0) == (r.cin % 32 == 0)
             for h in range(4, 2 * res + 1, 2) if h != r.H and c * h * h <= r.cin * res * res]
    return [max(cands)[1:] if cands else (r.cin, r.H)] + ([(r.cin, r.H)] if r.up else [])


@pytest.mark.gpu
@pytest.mark.parametrize('r', ROWS, ids=[r.id for r in ROWS])
def test_conv_row(cuda_device, r):
    t0 = time.perf_counter()
    dev = cuda_device
    seed = ROWS.index(r)
    m = make_layer(r.cin, r.cout, r.up, seed, nonsep=r.nonsep, demod=r.demod).to(dev)
    m.conv.precision = r.precision
    gen = torch.Generator().manual_seed(seed)
    ro = 2 * r.H if r.up else r.H
    x = torch.randn(r.B, r.cin, r.H, r.H, generator=gen).to(dev)
    style = torch.randn(r.B, STYLE_DIM, generator=gen).to(dev)
    noise = torch.randn(r.B, 1, ro, ro, generator=gen).to(dev)
    with torch.no_grad():
        got, kernels = launched_conv_kernels(lambda: m.conv(x, style))
        got_sty = m(x, style, noise=noise)
        # stale scratch: poison the layer scratch at the same batch without growing it, then run the row again
        for cin_p, h_p in poison_shapes(r):
            p = make_layer(cin_p, r.cout, r.up, seed + 1000, nonsep=r.nonsep, demod=r.demod).to(dev)
            p.conv.precision = r.precision
            px = torch.randn(r.B, cin_p, h_p, h_p, device=dev) * 1e6
            pout = p.conv(px, torch.randn(r.B, STYLE_DIM, device=dev))
            assert bool(torch.isfinite(pout).all()) and float(pout.abs().max()) > 1e4
        again = m.conv(x, style)
    torch.cuda.synchronize()
    ref, rss = restate(x, style, *conv_params(m))
    tau = TAU['fp32'] if SIMT in r.kernels else TAU[r.precision]
    err = normalised_error(got, ref, rss)
    sty_ref, mag = restate_styled(ref, noise, m.noise.weight.detach(), m.activate.bias.detach())
    sty_bound = math.sqrt(2.0) * (tau * rss + 8 * 2.0 ** -24 * mag)
    sty_err = float(((got_sty.double() - sty_ref).abs() / sty_bound).max())
    print(f'\n[{r.id}] B={r.B} {r.cin}->{r.cout} {r.H}^2{" up" if r.up else ""} {r.precision}: '
          f'max |err|/rss {err:.2e} (tau {tau:.0e}), styled {sty_err:.2f} of bound; '
          f'kernels {sorted(kernels)}; {time.perf_counter() - t0:.2f} s')
    assert got.shape == ref.shape and err <= tau, (r.id, err)
    assert sty_err <= 1.0, (r.id, sty_err)
    assert torch.equal(again, got), (r.id, 'differs after a call that left other data in the scratch')
    assert kernels == r.kernels, (r.id, sorted(kernels), sorted(r.kernels))
    if SIMT in r.kernels:
        assert not any(k.startswith('modconv_tc') or k.startswith('blur_act_split') for k in kernels)
