#!/usr/bin/env python
"""Multi-GPU self-consistency: the edge-sharded fit (torchrun, NCCL) must equal the
single-device fit on the same inputs (SURVEY 8e).  Run under torchrun."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import fcdiff_b200 as fcdiff                # noqa: E402
from fcdiff_b200 import dist as fdist       # noqa: E402
from oracle import iar_oracle as O          # noqa: E402


def run(b, bt, shards, device_shards=False, n_edges=None):
    fit = fcdiff.fit.UnsharedRegionFit()
    fit.model = fcdiff.UnsharedRegionModel()
    fit.model.eta += 0.1
    fit.b, fit.bt = b, bt
    fit.shards = shards
    fit.n_edges = n_edges
    fit.max_iters = 4
    fit.run()
    return fit


def main():
    shards = fdist.init_from_env("nccl")
    rank = dist.get_rank()
    ok = True
    for (N, H, U) in [(10, 20, 20), (33, 17, 31), (90, 50, 50)]:
        (_, _, _, _, b, bt) = O.sample(O.Theta(), N, H, U, np.random.RandomState(N))
        single = run(b, bt, None)
        sharded = run(b, bt, shards)                         # full host arrays on every rank
        C = b.shape[0]
        (c0, Cl) = shards.span(C)
        dev = run(torch.from_numpy(b[c0:c0 + Cl]).cuda(), torch.from_numpy(bt[c0:c0 + Cl]).cuda(), shards,
                  device_shards=True, n_edges=C)             # device edge shards + all-to-all re-layout
        for name, f in (("host-sharded", sharded), ("device-sharded", dev)):
            e = np.max(np.abs(np.array(f.energy) / np.array(single.energy) - 1))
            dF = np.max(np.abs(f._lq_F - single._lq_F))
            dR = np.max(np.abs(f._lq_R - single._lq_R))
            dth = max(abs(f.model.pi - single.model.pi), abs(f.model.eta - single.model.eta),
                      abs(f.model.epsilon - single.model.epsilon))
            good = e < 1e-9 and dF < 1e-7 and dR < 1e-7 and dth < 1e-9 and len(f.energy) == len(single.energy)
            ok = ok and good
            if rank == 0:
                print("N=%d %s: iters %d energy rel %.2e  lqF %.2e  lqR %.2e  theta %.2e  %s"
                      % (N, name, len(f.energy) - 1, e, dF, dR, dth, "OK" if good else "MISMATCH"), flush=True)
    # replica sweep: 5 labellings split over the ranks, gathered at the end, equal to rank-local runs
    from fcdiff_b200 import sweep
    (_, _, _, _, b, bt) = O.sample(O.Theta(), 12, 14, 10, np.random.RandomState(3))
    corr = np.concatenate([b, bt], axis=1)
    labels = np.r_[np.zeros(14, bool), np.ones(10, bool)]
    opts = dict(max_iters=3, rel_tol=-1.0)
    res = sweep.permutation_sweep(corr, labels, 4, seed=7, fit_options=opts, rank=rank, world=dist.get_world_size())
    ref = sweep.permutation_sweep(corr, labels, 4, seed=7, fit_options=opts, gather=False)
    good = sorted(res) == sorted(ref) and all(res[i]["energy"] == ref[i]["energy"] for i in ref)
    ok = ok and good
    if rank == 0:
        print("replica sweep over %d ranks: %s" % (dist.get_world_size(), "OK" if good else "MISMATCH"))
    t = torch.tensor([1.0 if ok else 0.0], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("DIST_CHECK", "PASS" if t.item() > 0 else "FAIL")
    dist.destroy_process_group()
    sys.exit(0 if t.item() > 0 else 1)


if __name__ == "__main__":
    main()
