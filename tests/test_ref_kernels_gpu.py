"""GPU parity against the REFERENCE'S OWN CUDA kernels (fused_bias_act_kernel.cu, upfirdn2d_kernel.cu).  Bit-exact:
same arithmetic, same FMA chain order.

The reference tree is not part of this repository, so what its kernels return on the seeded inputs below is recorded in
tests/golden/golden_ref_kernels_v1.npz (tests/golden/make_golden_ref_kernels.py): per case the output shape, a SHA-256
digest of the full output and a seeded sample of its values.  The vectors were recorded from this project's kernels,
which this test had found bit-equal to the reference's kernels compiled by oracle/build_ref.py; where oracle/_ref is
built, the recorder asserts that equality again before it writes.  The CPU test at the end ties the recorded samples to
the oracle's restatement of the two ops, so the recording cannot drift from the reference's algorithm unnoticed."""
import hashlib
import os

import numpy as np
import pytest
import torch

from oracle import stylegan2_oracle as so
from synthesis_in_style_b200.op import fused_bias_act, upfirdn2d_op

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'golden_ref_kernels_v1.npz')
SAMPLE = 512

FUSED_SHAPES = [(32, 512), (2, 128, 64, 64), (3, 5, 7, 9)]
FUSED_CODES = [(3, 0), (3, 1), (1, 0)]
UPFIRDN_CFGS = [
    # (major, H, W, up, down, pad, k)  the reference's six modes
    (64, 65, 65, 1, 1, (1, 1), 4), (7, 33, 20, 1, 1, (1, 1), 3), (6, 32, 32, 2, 1, (2, 1), 4),
    (6, 16, 16, 2, 1, (1, 0), 2), (5, 64, 64, 1, 2, (1, 1), 4), (5, 32, 32, 1, 2, (0, 0), 2),
    # planes of <= 32 x 32 outputs: the plane-group kernel (several planes per block, ragged last group, cropping pads)
    (300, 8, 8, 1, 1, (1, 1), 4), (64, 33, 33, 1, 1, (1, 1), 4), (1301, 4, 4, 2, 1, (2, 1), 4), (50, 8, 8, 2, 1, (2, 1), 4),
    (40, 16, 16, 1, 2, (1, 1), 4), (9, 20, 12, 1, 1, (-1, 2), 3), (33, 9, 9, 1, 1, (2, 2), 4)]


def fused_case(shape, code):
    """Key and CPU arguments of one fused_bias_act case."""
    g = torch.Generator().manual_seed(1)
    x = torch.randn(*shape, generator=g)
    b = torch.randn(shape[1], generator=g)
    r = torch.randn(*shape, generator=g) if code[1] == 1 else x.new_empty(0)
    return f'fused/{shape}/{code}', (x, b, r, code[0], code[1], 0.2, 2 ** 0.5)


def upfirdn_case(cfg):
    """Key and CPU arguments of one upfirdn2d case."""
    major, h, w, up, down, pad, ks = cfg
    g = torch.Generator().manual_seed(2)
    x = torch.randn(major, h, w, 1, generator=g)
    k = torch.randn(ks, ks, generator=g) if ks != 4 else so.make_kernel([1, 3, 3, 1]) * 4
    return f'upfirdn2d/{cfg}', (x, k, up, up, down, down, pad[0], pad[1], pad[0], pad[1])


def on_device(args, dev):
    return [a.to(dev) if torch.is_tensor(a) else a for a in args]


def digest(y):
    """SHA-256 of the float32 bytes, -0.0 folded into +0.0 (torch.equal does not tell them apart either)."""
    return np.frombuffer(hashlib.sha256((y.detach().cpu().contiguous() + 0.0).numpy().tobytes()).digest(), dtype=np.uint8)


def record(key, y):
    flat = y.detach().cpu().reshape(-1)
    idx = np.sort(np.random.RandomState(0).choice(flat.numel(), size=min(SAMPLE, flat.numel()), replace=False))
    return {f'{key}/shape': np.array(y.shape, dtype=np.int64), f'{key}/idx': idx.astype(np.int64),
            f'{key}/val': flat[torch.from_numpy(idx)].numpy(), f'{key}/sha256': digest(y)}


@pytest.fixture(scope='module')
def recorded():
    with np.load(GOLDEN) as z:
        return {k: z[k] for k in z.files}


def check(recorded, key, got):
    got = got.cpu()
    assert list(got.shape) == recorded[f'{key}/shape'].tolist(), key
    sample = got.reshape(-1)[torch.from_numpy(recorded[f'{key}/idx'])]
    assert torch.equal(sample, torch.from_numpy(recorded[f'{key}/val'])), f'{key}: sampled values differ from the reference kernel'
    assert np.array_equal(digest(got), recorded[f'{key}/sha256']), f'{key}: output differs from the reference kernel'


@pytest.mark.gpu
@pytest.mark.parametrize('shape', FUSED_SHAPES)
@pytest.mark.parametrize('code', FUSED_CODES)
def test_fused_bias_act_equals_reference_kernel(cuda_device, recorded, shape, code):
    key, args = fused_case(shape, code)
    check(recorded, key, fused_bias_act(*on_device(args, cuda_device)))


@pytest.mark.gpu
@pytest.mark.parametrize('cfg', UPFIRDN_CFGS)
def test_upfirdn2d_equals_reference_kernel(cuda_device, recorded, cfg):
    key, args = upfirdn_case(cfg)
    check(recorded, key, upfirdn2d_op(*on_device(args, cuda_device)))


def test_recorded_reference_kernel_outputs_follow_the_oracle(recorded):
    cases = [(fused_case(s, c), so.fused_bias_act) for s in FUSED_SHAPES for c in FUSED_CODES]
    cases += [(upfirdn_case(cfg), so.upfirdn2d_op) for cfg in UPFIRDN_CFGS]
    for (key, args), oracle_op in cases:
        want = oracle_op(*args)
        assert list(want.shape) == recorded[f'{key}/shape'].tolist(), key
        sample = want.reshape(-1)[torch.from_numpy(recorded[f'{key}/idx'])]
        torch.testing.assert_close(torch.from_numpy(recorded[f'{key}/val']), sample, rtol=1e-5, atol=1e-5, msg=key)
