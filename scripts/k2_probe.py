#!/usr/bin/env python
"""K2 in isolation on FIXED inputs: config 3 fitted for a few iterations, then the coded E-step launched
repeatedly on the state the last M-step left (same code plane, same records) -- timings that do not depend on
the fit's trajectory.  usage: python scripts/k2_probe.py [iters ...]"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import fcdiff_b200 as fcdiff  # noqa: E402


def main():
    iters = [int(a) for a in sys.argv[1:]] or [2, 8]
    (N, H, U) = (400, 500, 500)
    model = fcdiff.UnsharedRegionModel()
    (_, _, _, _, b, bt) = model.sample_device(N, H, U)
    for it in iters:
        f = fcdiff.fit.UnsharedRegionFit()
        f.model = fcdiff.UnsharedRegionModel()
        f.model.eta += 0.1
        (f.b, f.bt) = (b, bt)
        f.max_iters = it
        f.rel_tol = -1.0
        f.run()
        inp = f._in
        cnt = inp['bk_counts'].cpu().numpy().reshape(-1, 2) if 'bk_counts' in inp else None
        if cnt is not None:
            print("after %d iterations: full records %d (rows with any %d, unpeaked rows %d), half records %d (rows > 64: %d)" % (
                it, int(cnt[:, 0][cnt[:, 0] != 3 * U].sum()), int(((cnt[:, 0] > 0) & (cnt[:, 0] != 3 * U)).sum()),
                int((cnt[:, 0] == 3 * U).sum()), int(cnt[:, 1].sum()), int((cnt[:, 1] > 64).sum())))
        ms = []
        for r in range(40):
            (e0, e1) = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            e0.record()
            f._update_lq_F()
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        ms = sorted(ms[4:])
        print("  iters %d  K2 min %.4f  median %.4f ms" % (it, ms[0], ms[len(ms) // 2]))


if __name__ == "__main__":
    main()
