#!/usr/bin/env python
"""K1 timing on the GPU box: the tensor-core Gram vs the SIMT fp64-accumulate Gram at the config-3 shape.
(Accuracy of both paths, their agreement and the full-tile form are tested in tests/test_gpu_corr_edges.py
and tests/test_gpu_sampler_corr.py.)"""
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from fcdiff_b200 import corr          # noqa: E402


def run(ts_dev, fisher, simt):
    if simt:
        os.environ["FCD_CORR_SIMT"] = "1"
    else:
        os.environ.pop("FCD_CORR_SIMT", None)
    out = corr.correlations_device(ts_dev, fisher=fisher)
    torch.cuda.synchronize()
    return out


def main():
    # timing at config-3 shape (a slice of the subjects)
    (S, N, T) = (200, 400, 1200)
    ts_dev = torch.randn((S, N, T), dtype=torch.float32, device="cuda")
    for simt in (False, True):
        run(ts_dev, True, simt)
        t0 = time.perf_counter()
        for _ in range(3):
            run(ts_dev, True, simt)
        dt = (time.perf_counter() - t0) / 3
        print("%s: S=%d N=%d T=%d  %.2f ms  (%.1f subjects/ms)" % ("simt" if simt else "tc  ", S, N, T, dt * 1e3, S / (dt * 1e3)))


if __name__ == "__main__":
    main()
