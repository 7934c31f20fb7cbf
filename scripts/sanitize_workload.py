#!/usr/bin/env python
"""Small end-to-end workload for scripts/sanitize.sh: every kernel family of the hot path on
BASELINE.json configs 1-2 (reduced so that compute-sanitizer finishes in minutes)."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import fcdiff_b200 as fcdiff                      # noqa: E402
from fcdiff_b200 import corr                      # noqa: E402


def problem(N, H, U, seed):
    m = fcdiff.UnsharedRegionModel()
    m.rng = np.random.RandomState(seed)
    (_, _, _, _, b, bt) = m.sample(N, H, U)
    return b, bt


def one_fit(b, bt, shards=None, **opts):
    fit = fcdiff.fit.UnsharedRegionFit()
    fit.model = fcdiff.UnsharedRegionModel()
    fit.model.eta += 0.1
    fit.b, fit.bt = b, bt
    fit.shards = shards
    fit.max_iters = 3
    for (k, v) in opts.items():
        setattr(fit, k, v)
    fit.run()
    assert np.all(np.isfinite(fit.energy)), fit.energy
    return fit


def main():
    dist_mode = "--dist" in sys.argv
    shards = None
    if dist_mode:
        from fcdiff_b200 import dist as fdist
        shards = fdist.init_from_env("nccl")
    # config 1; a cut of config 2 (AAL-90); 70 regions: the blocked region sweep (N >= 64: cp.async tiles, L2 bulk
    # prefetch, double-buffered shared-memory tiles between the solver warp and the helper warps)
    for (N, H, U) in ((10, 20, 20), (40, 50, 50), (70, 12, 16)):
        (b, bt) = problem(N, H, U, N)
        one_fit(b, bt, shards)
        if dist_mode:
            continue
        one_fit(b, bt, edge_lookup="symmetric")
        one_fit(b, bt, elm_path="tiered", coded_estep=False)
        one_fit(b, bt, elm_path="streams")
        one_fit(b, bt, update_mu_sigma=True, edge_lookup="symmetric")
        for solver in ("newton",):
            if hasattr(fcdiff.fit.UnsharedRegionFit(), "theta_solver"):
                one_fit(b, bt, theta_solver=solver)
    if not dist_mode:
        ts = np.random.RandomState(0).standard_normal((4, 90, 200)).astype(np.float32)      # config 2's K1 shape
        z = corr.correlations(ts)
        assert np.all(np.isfinite(z))
        # persistent tcgen05 Gram kernel: a 16-row tail block (transposed tiles), a lone subject in the last pair,
        # both TMEM buffers reused
        ts = np.random.RandomState(2).standard_normal((5, 144, 96)).astype(np.float32)
        assert np.all(np.isfinite(corr.correlations(ts)))
        ts = np.random.RandomState(1).standard_normal((3, 20, 64)).astype(np.float32)       # SIMT Gram path
        assert np.all(np.isfinite(corr.correlations(ts, fisher=False)))
    torch.cuda.synchronize()
    if dist_mode:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    print("sanitize workload ok")


if __name__ == "__main__":
    main()
