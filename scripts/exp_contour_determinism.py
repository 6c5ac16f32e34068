"""Run the device contour stage repeatedly on the same masks (fresh stage / workspace each time) and compare outputs."""
import os, sys
import numpy, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'scripts'))
from synthesis_in_style_b200 import contours as pc, contours_device as pd
from contour_stage_bench import smooth_argmax_masks, COLORS
dev = torch.device('cuda:0')
for size, sig in ((128, (3, 3, 1, 1)), (256, (3, 3, 1, 1)), (256, (6, 6, 2.5, 2.5))):
    cfg = pc.ContourConfig(size, COLORS, ['8', '9'], ['12', '13'], True, 10)
    stacked = smooth_argmax_masks(8, size, sig, dev, 5)
    ref = None
    diffs = 0
    for it in range(12):
        stage = pd.DeviceContourStage(cfg)
        if it % 2:
            torch.empty(64 << 20, dtype=torch.uint8, device=dev).fill_(it * 37 % 251)     # churn the allocator
        out, flags = stage.run(stacked)
        torch.cuda.synchronize()
        cur = (out.cpu().numpy(), flags.cpu().numpy(), stage.last_info)
        if ref is None:
            ref = cur
        else:
            same = numpy.array_equal(cur[0], ref[0]) and numpy.array_equal(cur[1], ref[1]) and cur[2] == ref[2]
            diffs += not same
            if not same:
                print('  differs at it', it, 'pixels', int((cur[0] != ref[0]).any(-1).sum()), 'flags', cur[1].tolist(), ref[1].tolist(), cur[2], ref[2])
    print('size', size, sig, 'runs differing', diffs, 'info', ref[2])
