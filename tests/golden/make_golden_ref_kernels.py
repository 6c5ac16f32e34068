"""Record golden_ref_kernels_v1.npz: what the reference's own fused_bias_act / upfirdn2d CUDA kernels return on the
seeded cases of tests/test_ref_kernels_gpu.py (output shape, SHA-256 of the full output, a seeded sample of values).

Needs a CUDA device: `python tests/golden/make_golden_ref_kernels.py [OUT.npz]`.  The outputs are computed by this
project's two ops.  Where oracle/_ref holds the reference's kernels (oracle/build_ref.py), the script ASSERTS that both
agree bit for bit on every case before it writes, so the file stands in for the reference kernels where they are absent.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

import test_ref_kernels_gpu as t  # noqa: E402
from bench import load_ref_kernels  # noqa: E402
from synthesis_in_style_b200.op import fused_bias_act, upfirdn2d_op  # noqa: E402


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, 'golden_ref_kernels_v1.npz')
    dev = torch.device('cuda:0')
    ref = load_ref_kernels()
    cases = [(t.fused_case(s, c), fused_bias_act, 'ref_fused', 'fused_bias_act') for s in t.FUSED_SHAPES for c in t.FUSED_CODES]
    cases += [(t.upfirdn_case(cfg), upfirdn2d_op, 'ref_upfirdn2d', 'upfirdn2d') for cfg in t.UPFIRDN_CFGS]
    out = {}
    for (key, args), op, ref_mod, ref_fn in cases:
        args = t.on_device(args, dev)
        got = op(*args)
        if ref is not None:
            want = getattr(ref[ref_mod], ref_fn)(*args)
            assert got.shape == want.shape and torch.equal(got, want), f'{key}: differs from the reference kernel'
        out.update(t.record(key, got))
    np.savez_compressed(path, **out)
    print(f'wrote {path}: {len(cases)} cases, {os.path.getsize(path) / 1024:.1f} KiB, '
          f'{"checked against" if ref is not None else "without"} the reference kernels')


if __name__ == '__main__':
    main()
