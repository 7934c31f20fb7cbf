#!/usr/bin/env python
"""
Partial correlations (fcd_corr_partial) on the K1 workload's planted 8-factor series, generated on the device
from a seed: 1000 subjects x 400 regions x 1200 frames, the same with 200 frames (fewer frames than regions)
and 2000 x 1000 x 1200.  Inputs are 1.9 - 9.6 GB, beyond the 126 MB of L2.

Per shape: the call's time from CUDA events after a warm-up call (Ledoit-Wolf, Fisher z), the Pearson path
(fcd_corr_fisherz) on the same series, and the per-stage device time of one call from torch.profiler in a
separate pass -- standardise (standardise_kernel), Gram (partial_gram_kernel, frame_sq_kernel), shrink
(partial_shrink_kernel), factor and inverse (partial_invert_kernel), epilogue (partial_epilogue_kernel).
fp64 FMAs from the shapes (Gram S N^2 T / 2, inverse S N^3 / 2) give the achieved fp64 FLOP/s of those
stages and of the call.  The card's name and power limit are read in the same run.  Prints one JSON line.

    python scripts/partial_corr_bench.py [--reps 3] [--seed 1] [--shapes 1000x400x1200,...]
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from fcdiff_b200 import corr                    # noqa: E402
from clean_corr_bench import card, timed, workload    # noqa: E402

STAGES = (("standardise_kernel", "standardise"), ("clean_kernel", "standardise"), ("confound_basis", "standardise"),
          ("partial_gram_kernel", "gram"), ("frame_sq_kernel", "gram"), ("partial_shrink_kernel", "shrink"),
          ("partial_invert_kernel", "invert"), ("partial_epilogue_kernel", "epilogue"), ("mark_status", "epilogue"))


def stage_split(fn):
    """Per-stage device time (ms) of one call, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if t <= 0:
            continue
        for (key, stage) in STAGES:
            if key in ev.key:
                out[stage] = out.get(stage, 0.0) + t / 1000.0
                break
    return out


def run(S, N, T, reps, seed):
    C = N * (N - 1) // 2
    (ts, _) = workload(S, N, T, seed)
    out = torch.empty((C, S), dtype=torch.float64, device="cuda")
    delta = torch.empty((S,), dtype=torch.float64, device="cuda")

    def partial():
        corr.correlations_device(ts, fisher=True, out=out, kind="partial", shrinkage_out=delta)

    def pearson():
        corr.correlations_device(ts, fisher=True, out=out)

    ms_p = timed(partial, reps)
    ms_r = timed(pearson, reps)
    split = stage_split(partial)
    fma_gram = S * N * N * T / 2.0
    fma_inv = S * N ** 3 / 2.0
    res = {"shape": [S, N, T], "partial_ms": ms_p, "pearson_ms": ms_r, "stages_ms": split,
           "fma_gram": fma_gram, "fma_invert": fma_inv,
           "call_fp64_TFLOPs": 2.0 * (fma_gram + fma_inv) / (ms_p * 1e-3) / 1e12,
           "delta_median": float(delta.median())}
    if split.get("gram"):
        res["gram_fp64_TFLOPs"] = 2.0 * fma_gram / (split["gram"] * 1e-3) / 1e12
    if split.get("invert"):
        res["invert_fp64_TFLOPs"] = 2.0 * fma_inv / (split["invert"] * 1e-3) / 1e12
    res["finite"] = bool(torch.isfinite(out).all())
    del ts, out
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--shapes", default="1000x400x1200,1000x400x200,2000x1000x1200")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("partial_corr_bench.py needs a CUDA device")
    res = {"card": card(), "workload": "planted 8-factor series (seed %d), Ledoit-Wolf, Fisher z" % args.seed,
           "runs": []}
    for sh in args.shapes.split(","):
        (S, N, T) = (int(v) for v in sh.split("x"))
        res["runs"].append(run(S, N, T, args.reps, args.seed))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
