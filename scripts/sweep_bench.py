"""Timing of the region sweep (fcd_estep_qR) on one GPU at the shapes the bench meets, in the launch shape the
code chooses from the region and patient counts.
    python scripts/sweep_bench.py                # table to stdout
    python scripts/sweep_bench.py 400x63 1131x63 # only these (regions x patients) shapes
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from fcdiff_b200 import _dev, _lib      # noqa: E402

SHAPES = [(400, 500), (400, 63), (566, 250), (800, 125), (1131, 63), (1000, 1000), (1000, 125)]


def main(shapes):
    lib = _lib.load()
    print("%-22s %12s   %s" % ("N, patients, regime", "time", "checksum"))
    for (N, Ul) in shapes:
        C = N * (N - 1) // 2
        for (regime, scale) in (("undecided", 0.02), ("decided", 3.0)):
            g = torch.Generator(device="cuda").manual_seed(N + Ul)
            WT = scale * torch.randn((Ul * C * 2,), dtype=torch.float64, device="cuda", generator=g)
            q0 = torch.rand((N * Ul,), dtype=torch.float64, device="cuda", generator=g)
            q = torch.stack([q0, 1.0 - q0], dim=1).reshape(-1).contiguous()
            lq = torch.zeros_like(q)
            lp = _lib.d3(np.log(np.array([0.7, 0.3])))
            st = _dev.stream()

            def run():
                _lib.check(lib.fcd_estep_qR(_dev.ptr(WT), C, N, Ul, 0, Ul, lp, 0, _dev.ptr(q), _dev.ptr(lq), st),
                           "fcd_estep_qR")
            for _ in range(3):
                run()
            (e0, e1) = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            R = 10 if C * Ul < 2e8 else 4
            torch.cuda.synchronize()
            e0.record()
            for _ in range(R):
                run()
            e1.record()
            torch.cuda.synchronize()
            print("%-22s %9.1f us   %.6f" % ("%d, %d, %s" % (N, Ul, regime), e0.elapsed_time(e1) / R * 1e3,
                                             float(q.reshape(-1, 2)[:, 0].sum().item())))
            del WT, q, lq


if __name__ == "__main__":
    main([tuple(int(v) for v in a.split("x")) for a in sys.argv[1:]] or SHAPES)
